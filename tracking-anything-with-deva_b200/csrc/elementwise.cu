// HBM-bound helper kernels of the NHWC fp16 network path: layout/precision conversion at the API boundary,
// max-pool, bilinear x2 + skip add, area down-sampling, CBAM (reference deva/model/cbam.py:21-77), the
// non-standard sensory GRU (modules.py:145-149), and the soft-aggregation / x4 upsampling / softmax tail
// (network.py:33-40,144-168).  One thread per output element (or per pixel x channel-vector); all accesses
// are coalesced along the channel axis.
#include <cuda_fp16.h>
#include <math_constants.h>
#include <stdint.h>

#include "common.h"
#include "elementwise.h"

namespace b200 {
namespace ew {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ void ld8(const __half* p, float (&f)[8]) {
  const uint4 v = *reinterpret_cast<const uint4*>(p);
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e) { const float2 t = __half22float2(h[e]); f[2 * e] = t.x; f[2 * e + 1] = t.y; }
}
__device__ __forceinline__ void st8(__half* p, const float (&f)[8], bool relu) {
  uint4 v;
  __half2* h = reinterpret_cast<__half2*>(&v);
#pragma unroll
  for (int e = 0; e < 4; ++e)
    h[e] = relu ? __floats2half2_rn(fmaxf(f[2 * e], 0.f), fmaxf(f[2 * e + 1], 0.f)) : __floats2half2_rn(f[2 * e], f[2 * e + 1]);
  *reinterpret_cast<uint4*>(p) = v;
}

// ---------------------------------------------------------------- layout conversion
// fp32 NCHW [B,C,H,W] -> fp16 NHWC [B,H,W,Cp] (channels >= C are zero)
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, __half* __restrict__ dst, int B, int C, int H, int W,
                                    int Cp) {
  const long long total = (long long)B * H * W * Cp;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % Cp);
    long long p = i / Cp;
    const int x = (int)(p % W); p /= W;
    const int y = (int)(p % H);
    const int b = (int)(p / H);
    dst[i] = (c < C) ? __float2half_rn(src[(((long long)b * C + c) * H + y) * W + x]) : __float2half_rn(0.f);
  }
}
// fp16 NHWC [B,H,W,C] -> fp32 NCHW [B,C,H,W]
__global__ void nhwc_to_nchw_kernel(const __half* __restrict__ src, float* __restrict__ dst, int B, int C, int H, int W) {
  const long long total = (long long)B * C * H * W;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int x = (int)(i % W);
    long long p = i / W;
    const int y = (int)(p % H); p /= H;
    const int c = (int)(p % C);
    const int b = (int)(p / C);
    dst[i] = __half2float(src[(((long long)b * H + y) * W + x) * C + c]);
  }
}
// im2col for the 7x7 stride-2 pad-3 stems (resnet.py:120): planes fp32 [B, C, H, W] -> fp16 [B, H/2, W/2, Kp]
// with column k = (kh*7 + kw)*C + c for k < 49*C and zeros up to Kp (a multiple of 64).  The stem then runs
// as a 1x1 implicit GEMM over Kp "channels" on the tensor cores.
constexpr int IM_XT = 64;  // output columns per block
__global__ void __launch_bounds__(256)
stem_im2col_kernel(const float* __restrict__ src, __half* __restrict__ dst, __half* __restrict__ dst_lo,
                   int B, int C, int H, int W, int Kp) {
  // Block = (image b, output row yo, IM_XT output columns).  The 7 input rows x (2*IM_XT + 5) input columns of all C
  // planes are staged in shared memory with coalesced loads; each thread then emits 8 consecutive im2col columns
  // (one 16-byte store for the fp16 values, one for the remainders).
  extern __shared__ float patch[];  // [C][7][PW]
  const int Ho = H / 2, Wo = W / 2;
  constexpr int PW = 2 * IM_XT + 5;
  const int b = blockIdx.y / Ho, yo = blockIdx.y - b * Ho;
  const int xo0 = blockIdx.x * IM_XT;
  const int x_in0 = 2 * xo0 - 3, y_in0 = 2 * yo - 3;
  const float* img = src + (long long)b * C * H * W;
  for (int i = threadIdx.x; i < C * 7 * PW; i += 256) {
    const int px = i % PW, r = (i / PW) % 7, c = i / (7 * PW);
    const int y = y_in0 + r, x = x_in0 + px;
    patch[i] = (y >= 0 && y < H && x >= 0 && x < W) ? img[((long long)c * H + y) * W + x] : 0.f;
  }
  __syncthreads();
  const int nx = min(IM_XT, Wo - xo0);
  const long long out_base = (((long long)b * Ho + yo) * Wo + xo0) * Kp;
  const int kreal = 49 * C, K8 = Kp / 8;
  for (int i = threadIdx.x; i < nx * K8; i += 256) {
    const int xl = i / K8, k0 = (i - xl * K8) * 8;
    float v[8], r[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = k0 + e;
      float x = 0.f;
      if (k < kreal) {
        const int tap = k / C, c = k - tap * C;
        const int ky = tap / 7, kx = tap - ky * 7;
        x = patch[(c * 7 + ky) * PW + 2 * xl + kx];
      }
      v[e] = x;
      r[e] = x - __half2float(__float2half_rn(x));
    }
    st8(dst + out_base + (long long)xl * Kp + k0, v, false);
    if (dst_lo) st8(dst_lo + out_base + (long long)xl * Kp + k0, r, false);
  }
}

// Pixel-per-thread variant for the shapes the network uses (C = 1: mask planes, Kp = 64; C = 3: image, Kp = 192, with
// or without the fp16 remainders).  The generic kernel spends ~120 instructions of index arithmetic per 16-byte store
// and ran at 16-28 % of the HBM peak; here a thread owns one output pixel, reads its 49*C taps from a patch staged in
// shared memory (even / odd input columns de-interleaved so consecutive pixels read consecutive words) with compile-time
// tap offsets, and writes its whole im2col row with 256-bit stores.  Same values as the generic kernel.
constexpr int IM1_XT = 128;
template <int C, int ROWS, bool LO>
__global__ void __launch_bounds__(IM1_XT)
stem_im2col_px_kernel(const float* __restrict__ src, __half* __restrict__ dst, __half* __restrict__ dst_lo, int B, int H, int W) {
  constexpr int PR = 2 * ROWS + 5;      // input rows under ROWS output rows
  constexpr int PH = IM1_XT + 3;        // input column x_in0 + 2*i (+1) for i in [0, PH)
  constexpr int KP = (49 * C + 63) / 64 * 64;
  __shared__ float pe[C][PR][PH], po[C][PR][PH];
  const int Ho = H / 2, Wo = W / 2;
  const int groups = (Ho + ROWS - 1) / ROWS;
  const int b = blockIdx.y / groups, yo0 = (blockIdx.y - b * groups) * ROWS;
  const int xo0 = blockIdx.x * IM1_XT;
  const int x_in0 = 2 * xo0 - 3, y_in0 = 2 * yo0 - 3;
  const float* img = src + (long long)b * C * H * W;
  for (int i = threadIdx.x; i < C * PR * 2 * PH; i += IM1_XT) {
    const int px = i % (2 * PH), r = (i / (2 * PH)) % PR, c = i / (2 * PH * PR);
    const int y = y_in0 + r, x = x_in0 + px;
    const float v = (y >= 0 && y < H && x >= 0 && x < W) ? img[((long long)c * H + y) * W + x] : 0.f;
    if (px & 1) po[c][r][px >> 1] = v;
    else pe[c][r][px >> 1] = v;
  }
  __syncthreads();
  const int xl = threadIdx.x, xo = xo0 + xl;
  if (xo >= Wo) return;
#pragma unroll 1
  for (int rr = 0; rr < ROWS; ++rr) {
    const int yo = yo0 + rr;
    if (yo >= Ho) break;
    const long long out = (((long long)b * Ho + yo) * Wo + xo) * KP;
#pragma unroll
    for (int k0 = 0; k0 < KP; k0 += 16) {  // 16 columns = one 32-byte store (and one for the remainders)
      uint4 oh[2], ol[2];
      __half2* h2 = reinterpret_cast<__half2*>(oh);
      __half2* l2 = reinterpret_cast<__half2*>(ol);
#pragma unroll
      for (int k2 = 0; k2 < 8; ++k2) {
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int k = k0 + 2 * k2 + e;  // column k = (ky*7 + kx)*C + c
          if (k < 49 * C) {
            const int tap = k / C, c = k - tap * C, ky = tap / 7, kx = tap - ky * 7;
            v[e] = (kx & 1) ? po[c][2 * rr + ky][xl + (kx >> 1)] : pe[c][2 * rr + ky][xl + (kx >> 1)];
          } else {
            v[e] = 0.f;
          }
        }
        h2[k2] = __floats2half2_rn(v[0], v[1]);
        if (LO) {
          const float2 back = __half22float2(h2[k2]);
          l2[k2] = __floats2half2_rn(v[0] - back.x, v[1] - back.y);
        }
      }
      asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + out + k0), "r"(oh[0].x), "r"(oh[0].y),
                   "r"(oh[0].z), "r"(oh[0].w), "r"(oh[1].x), "r"(oh[1].y), "r"(oh[1].z), "r"(oh[1].w)
                   : "memory");
      if (LO)
        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst_lo + out + k0), "r"(ol[0].x),
                     "r"(ol[0].y), "r"(ol[0].z), "r"(ol[0].w), "r"(ol[1].x), "r"(ol[1].y), "r"(ol[1].z), "r"(ol[1].w)
                     : "memory");
    }
  }
}

// ---------------------------------------------------------------- pooling / resampling (NHWC fp16, 8 channels per thread)
// 3x3 stride-2 pad-1 max pool (resnet.py:123)
__global__ void maxpool_kernel(const __half* __restrict__ x, const __half* __restrict__ x_lo, __half* __restrict__ y,
                               __half* __restrict__ y_lo, int B, int H, int W, int C) {
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, C8 = C / 8;
  const long long total = (long long)B * Ho * Wo * C8;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % C8) * 8;
    long long p = i / C8;
    const int xo = (int)(p % Wo); p /= Wo;
    const int yo = (int)(p % Ho);
    const int b = (int)(p / Ho);
    float m[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) m[e] = -CUDART_INF_F;
    for (int dy = -1; dy <= 1; ++dy) {
      const int yy = 2 * yo + dy;
      if (yy < 0 || yy >= H) continue;
      for (int dx = -1; dx <= 1; ++dx) {
        const int xx = 2 * xo + dx;
        if (xx < 0 || xx >= W) continue;
        float f[8];
        const long long o = (((long long)b * H + yy) * W + xx) * C + c;
        ld8(x + o, f);
        if (x_lo) {
          float l[8];
          ld8(x_lo + o, l);
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] += l[e];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) m[e] = fmaxf(m[e], f[e]);
      }
    }
    const long long oo = (((long long)b * Ho + yo) * Wo + xo) * C + c;
    st8(y + oo, m, false);
    if (y_lo) {
      float r[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) r[e] = m[e] - __half2float(__float2half_rn(m[e]));
      st8(y_lo + oo, r, false);
    }
  }
}

// out = bilinear_x2(g) + skip (skip is one image broadcast over the batch); writes raw and/or relu
// (MaskUpsampleBlock: upsample_groups + distributor 'add', modules.py:88-91)
__global__ void __launch_bounds__(256)
up2_add_kernel(const __half* __restrict__ g, const __half* __restrict__ skip, __half* __restrict__ raw,
               __half* __restrict__ relu, int B, int h, int w, int C) {
  // blockIdx.y = (image, output row): the two source rows and their weights are uniform per block
  const int H = 2 * h, W = 2 * w, C8 = C / 8;
  const int b = blockIdx.y / H, Y = blockIdx.y - b * H;
  const float sy = fmaxf((Y + 0.5f) * 0.5f - 0.5f, 0.f);  // align_corners=False: src = (dst + 0.5)/2 - 0.5, clamped
  const int y0 = (int)sy, y1 = min(y0 + 1, h - 1);
  const float wy = sy - y0;
  const __half* r0 = g + ((long long)b * h + y0) * w * C;
  const __half* r1 = g + ((long long)b * h + y1) * w * C;
  const __half* sk = skip + (long long)Y * W * C;
  const long long obase = ((long long)b * H + Y) * W * C;
  const int row_vecs = W * C8;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < row_vecs; i += gridDim.x * 256) {
    const int X = i / C8, c = (i - X * C8) * 8;
    const float sx = fmaxf((X + 0.5f) * 0.5f - 0.5f, 0.f);
    const int x0 = (int)sx, x1 = min(x0 + 1, w - 1);
    const float wx = sx - x0;
    float a[8], bq[8], cq[8], d[8], o[8], s_[8];
    ld8(r0 + x0 * C + c, a);
    ld8(r0 + x1 * C + c, bq);
    ld8(r1 + x0 * C + c, cq);
    ld8(r1 + x1 * C + c, d);
    ld8(sk + X * C + c, s_);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float top = a[e] + (bq[e] - a[e]) * wx, bot = cq[e] + (d[e] - cq[e]) * wx;
      o[e] = top + (bot - top) * wy + s_[e];
    }
    const long long off = obase + X * C + c;
    if (raw) st8(raw + off, o, false);
    if (relu) st8(relu + off, o, true);
  }
}

// Split-precision twin (residual stream carried as fp16 hi/lo pairs, DESIGN section 4 "precision plan"): g = g + g_lo on
// input; the raw sum is written as (hi, lo), the ReLU'd copy - an MMA operand only - as hi.
__device__ __forceinline__ void st8_split(__half* hi, __half* lo, const float (&f)[8]) {
  uint4 vh, vl;
  __half2* h2 = reinterpret_cast<__half2*>(&vh);
  __half2* l2 = reinterpret_cast<__half2*>(&vl);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h2[e] = __floats2half2_rn(f[2 * e], f[2 * e + 1]);
    const float2 back = __half22float2(h2[e]);
    l2[e] = __floats2half2_rn(f[2 * e] - back.x, f[2 * e + 1] - back.y);
  }
  *reinterpret_cast<uint4*>(hi) = vh;
  *reinterpret_cast<uint4*>(lo) = vl;
}
__global__ void __launch_bounds__(256)
up2_add_split_kernel(const __half* __restrict__ g, const __half* __restrict__ g_lo, const __half* __restrict__ skip,
                     const __half* __restrict__ skip_lo, __half* __restrict__ raw, __half* __restrict__ raw_lo,
                     __half* __restrict__ relu, __half* __restrict__ relu_lo, unsigned char* __restrict__ relu_lo8, int B,
                     int h, int w, int C) {
  // A thread owns 8 channels of the 2 x 2 OUTPUT block {2k-1, 2k} x {2j-1, 2j}: with align_corners = False these four
  // pixels interpolate between the same four source pixels (rows k-1, k / columns j-1, j, clamped at the border) with
  // weights 0.25 / 0.75, so the source quad (hi + lo) is loaded once per four outputs and there is no serial walk:
  // every thread is one independent load -> compute -> store chain (the row-walking version kept the DRAM traffic at the
  // algorithmic 1x but ran at half the HBM rate: eight dependent rows per thread; the per-pixel version before it re-read
  // the source 5x).  blockIdx.y = (image, k), k in [0, h]; the clamped border blocks produce the reference's values
  // exactly (a + (a - a) * wx == a).
  const int H = 2 * h, W = 2 * w, C8 = C / 8;
  const int b = blockIdx.y / (h + 1), k = blockIdx.y - b * (h + 1);
  const int ya = max(k - 1, 0), yb = min(k, h - 1);
  const int row_vecs = (w + 1) * C8;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < row_vecs; i += gridDim.x * 256) {
    const int j = i / C8, c = (i - j * C8) * 8;
    const int xa = max(j - 1, 0), xb = min(j, w - 1);
    float qa[8], qb[8], qc[8], qd[8], l[8];  // source quad: (ya, xa), (ya, xb), (yb, xa), (yb, xb)
    const long long oa = (((long long)b * h + ya) * w) * C + c, ob = (((long long)b * h + yb) * w) * C + c;
    auto load = [&](const long long o, float (&q)[8]) {
      ld8(g + o, q);
      ld8(g_lo + o, l);
#pragma unroll
      for (int e = 0; e < 8; ++e) q[e] += l[e];
    };
    load(oa + (long long)xa * C, qa);
    load(oa + (long long)xb * C, qb);
    load(ob + (long long)xa * C, qc);
    load(ob + (long long)xb * C, qd);
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int Y = 2 * k - 1 + dy;
      if (Y < 0 || Y >= H) continue;
      const float wy = dy ? 0.75f : 0.25f;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int X = 2 * j - 1 + dx;
        if (X < 0 || X >= W) continue;
        const float wx = dx ? 0.75f : 0.25f;
        float o[8], s_[8];
        ld8(skip + ((long long)Y * W + X) * C + c, s_);
        if (skip_lo) {
          ld8(skip_lo + ((long long)Y * W + X) * C + c, l);
#pragma unroll
          for (int e = 0; e < 8; ++e) s_[e] += l[e];
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float top = qa[e] + (qb[e] - qa[e]) * wx, bot = qc[e] + (qd[e] - qc[e]) * wx;
          o[e] = top + (bot - top) * wy + s_[e];
        }
        const long long off = (((long long)b * H + Y) * W + X) * C + c;
        if (raw) st8_split(raw + off, raw_lo + off, o);
        if (relu_lo) {
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
          st8_split(relu + off, relu_lo + off, o);
        } else if (relu_lo8) {  // low-order part as e4m3 of (x - fp16(x)) * 4096: operand of an fp8 correction pass
          uint32_t w8[2];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
          st8(relu + off, o, false);
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            float q4[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) q4[t] = (o[4 * e + t] - __half2float(__float2half_rn(o[4 * e + t]))) * 4096.f;
            unsigned short a16, b16;
            asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(a16) : "f"(q4[1]), "f"(q4[0]));
            asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(b16) : "f"(q4[3]), "f"(q4[2]));
            w8[e] = (uint32_t)a16 | ((uint32_t)b16 << 16);
          }
          *reinterpret_cast<uint2*>(relu_lo8 + off) = make_uint2(w8[0], w8[1]);
        } else if (relu) {
          st8(relu + off, o, true);
        }
      }
    }
  }
}

// r x r average pooling (F.interpolate mode='area' with an integer ratio), NHWC fp16
__global__ void area_down_kernel(const __half* __restrict__ x, __half* __restrict__ y, int B, int H, int W, int C, int r) {
  const int Ho = H / r, Wo = W / r, C8 = C / 8;
  const long long total = (long long)B * Ho * Wo * C8;
  const float inv = 1.f / (r * r);
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int c = (int)(i % C8) * 8;
    long long p = i / C8;
    const int xo = (int)(p % Wo); p /= Wo;
    const int yo = (int)(p % Ho);
    const int b = (int)(p / Ho);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int dy = 0; dy < r; ++dy)
      for (int dx = 0; dx < r; ++dx) {
        float f[8];
        ld8(x + (((long long)b * H + yo * r + dy) * W + xo * r + dx) * C + c, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] += f[e];
      }
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] *= inv;
    st8(y + (((long long)b * Ho + yo) * Wo + xo) * C + c, acc, false);
  }
}
// same for single-channel fp32 planes [B,H,W] -> [B,H/r,W/r]
__global__ void area_down_plane_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W, int r) {
  const int Ho = H / r, Wo = W / r;
  const long long total = (long long)B * Ho * Wo;
  const float inv = 1.f / (r * r);
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int xo = (int)(i % Wo);
    long long p = i / Wo;
    const int yo = (int)(p % Ho);
    const int b = (int)(p / Ho);
    float acc = 0.f;
    for (int dy = 0; dy < r; ++dy)
      for (int dx = 0; dx < r; ++dx) acc += x[((long long)b * H + yo * r + dy) * W + xo * r + dx];
    y[i] = acc * inv;
  }
}

// ---------------------------------------------------------------- CBAM (cbam.py:21-77)
// per (image, channel) partial sum and max over a slice of the pixels.  grid (B, kPoolSplit), 256 threads: a thread owns
// 8 channels (one 16-byte load per pixel and operand) and every (256 / (C/8))-th pixel of the slice; the pixel lanes are
// folded through shared memory.  (The one-channel-per-thread version issued 2-byte loads: 64 bytes per warp instruction.)
constexpr int kPoolSplit = 64;
__global__ void __launch_bounds__(256)
cbam_pool_kernel(const __half* __restrict__ x, const __half* __restrict__ x_lo, float* __restrict__ psum,
                 float* __restrict__ pmax, int HW, int C) {
  __shared__ float ss[256 * 8], sm[256 * 8];
  const int b = blockIdx.x, sp = blockIdx.y;
  const int C8 = C / 8, lanes = 256 / C8;  // pixel lanes (host guarantees 256 % C8 == 0)
  const int cv = threadIdx.x % C8, pl = threadIdx.x / C8;
  const int per = (HW + kPoolSplit - 1) / kPoolSplit;
  const int i0 = sp * per, i1 = min(HW, i0 + per);
  float s[8], m[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) { s[e] = 0.f; m[e] = -CUDART_INF_F; }
  for (int i = i0 + pl; i < i1; i += lanes) {
    const long long o = ((long long)b * HW + i) * C + cv * 8;
    float v[8];
    ld8(x + o, v);
    if (x_lo) {
      float l[8];
      ld8(x_lo + o, l);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] += l[e];
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) { s[e] += v[e]; m[e] = fmaxf(m[e], v[e]); }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) { ss[e * 256 + threadIdx.x] = s[e]; sm[e * 256 + threadIdx.x] = m[e]; }
  __syncthreads();
  if (pl == 0) {
    for (int q = 1; q < lanes; ++q) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        s[e] += ss[e * 256 + q * C8 + cv];
        m[e] = fmaxf(m[e], sm[e * 256 + q * C8 + cv]);
      }
    }
    const long long o = ((long long)b * kPoolSplit + sp) * C + cv * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) { psum[o + e] = s[e]; pmax[o + e] = m[e]; }
  }
}
// gate[b,c] = sigmoid(mlp(avg) + mlp(max)), mlp = Linear(C,R) -> ReLU -> Linear(R,C); one block per image
__global__ void cbam_mlp_kernel(const float* __restrict__ psum, const float* __restrict__ pmax, int HW,
                                const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2,
                                const float* __restrict__ b2, float* __restrict__ gate, int C, int R) {
  extern __shared__ float sm[];  // avg[C] | max[C] | hid[2R]
  float* avg = sm;
  float* mx = sm + C;
  float* hid = sm + 2 * C;
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f, m = -CUDART_INF_F;
    for (int sp = 0; sp < kPoolSplit; ++sp) {
      s += psum[((long long)b * kPoolSplit + sp) * C + c];
      m = fmaxf(m, pmax[((long long)b * kPoolSplit + sp) * C + c]);
    }
    avg[c] = s / HW;
    mx[c] = m;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int r = warp; r < 2 * R; r += nwarp) {  // one warp per hidden unit: coalesced weight rows
    const float* src = (r < R) ? avg : mx;
    const float* wr = w1 + (long long)(r % R) * C;
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a += wr[c] * src[c];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) hid[r] = fmaxf(a + b1[r % R], 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 2.f * b2[c];
    for (int r = 0; r < R; ++r) a += w2[(long long)c * R + r] * (hid[r] + hid[R + r]);
    gate[b * C + c] = sigmoidf_(a);
  }
}
// per pixel: max and mean over channels of x * gate -> stats [B,HW,2]; one warp per pixel, 8 channels per lane and load
__global__ void cbam_stats_kernel(const __half* __restrict__ x, const __half* __restrict__ x_lo, const float* __restrict__ gate,
                                  float* __restrict__ stats, int B, int HW, int C) {
  const long long pix = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pix >= (long long)B * HW) return;
  const int b = (int)(pix / HW);
  const __half* p = x + pix * C;
  const __half* pl = x_lo ? x_lo + pix * C : nullptr;
  const float* g = gate + b * C;
  float s = 0.f, m = -CUDART_INF_F;
  for (int c = lane * 8; c < C; c += 256) {
    float v[8];
    ld8(p + c, v);
    if (pl) {
      float l[8];
      ld8(pl + c, l);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] += l[e];
    }
    const float4 g0 = *reinterpret_cast<const float4*>(g + c), g1 = *reinterpret_cast<const float4*>(g + c + 4);
    const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float t = v[e] * gg[e];
      s += t;
      m = fmaxf(m, t);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  }
  if (lane == 0) { stats[pix * 2] = m; stats[pix * 2 + 1] = s / C; }
}
// out = x + x * gate * sigmoid(conv7x7(stats))   (FeatureFusion: g + attention(g)); one warp per pixel
__global__ void cbam_apply_kernel(const __half* __restrict__ x, const float* __restrict__ gate, const float* __restrict__ stats,
                                  const float* __restrict__ ws, const float* __restrict__ bs, __half* __restrict__ raw,
                                  __half* __restrict__ relu, int B, int H, int W, int C) {
  const long long pix = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pix >= (long long)B * H * W) return;
  const int b = (int)(pix / ((long long)H * W));
  const int rem = (int)(pix - (long long)b * H * W);
  const int y = rem / W, xq = rem - y * W;
  float a = 0.f;
  for (int t = lane; t < 98; t += 32) {
    const int ch = t / 49, k = t % 49, dy = k / 7 - 3, dx = k % 7 - 3;
    const int yy = y + dy, xx = xq + dx;
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) a += ws[t] * stats[(((long long)b * H + yy) * W + xx) * 2 + ch];
  }
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  const float sg = sigmoidf_(a + bs[0]);
  const float* g = gate + b * C;
  for (int c = lane * 8; c < C; c += 256) {
    float v[8], o[8];
    ld8(x + pix * C + c, v);
#pragma unroll
    for (int e = 0; e < 8; ++e) o[e] = v[e] + v[e] * g[c + e] * sg;
    if (raw) st8(raw + pix * C + c, o, false);
    if (relu) st8(relu + pix * C + c, o, true);
  }
}

// split-precision twin of cbam_apply_kernel: x = x + x_lo on input, raw written as (hi, lo), relu as hi
__global__ void cbam_apply_split_kernel(const __half* __restrict__ x, const __half* __restrict__ x_lo,
                                        const float* __restrict__ gate, const float* __restrict__ stats,
                                        const float* __restrict__ ws, const float* __restrict__ bs,
                                        __half* __restrict__ raw, __half* __restrict__ raw_lo, __half* __restrict__ relu,
                                        __half* __restrict__ relu_lo, int B, int H, int W, int C) {
  const long long pix = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (pix >= (long long)B * H * W) return;
  const int b = (int)(pix / ((long long)H * W));
  const int rem = (int)(pix - (long long)b * H * W);
  const int y = rem / W, xq = rem - y * W;
  float a = 0.f;
  for (int t = lane; t < 98; t += 32) {
    const int ch = t / 49, k = t % 49, dy = k / 7 - 3, dx = k % 7 - 3;
    const int yy = y + dy, xx = xq + dx;
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) a += ws[t] * stats[(((long long)b * H + yy) * W + xx) * 2 + ch];
  }
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  const float sg = sigmoidf_(a + bs[0]);
  const float* g = gate + b * C;
  for (int c = lane * 8; c < C; c += 256) {
    float v[8], l[8], o[8];
    ld8(x + pix * C + c, v);
    ld8(x_lo + pix * C + c, l);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float t = v[e] + l[e];
      o[e] = t + t * g[c + e] * sg;
    }
    st8_split(raw + pix * C + c, raw_lo + pix * C + c, o);
    if (relu) {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = fmaxf(o[e], 0.f);
      if (relu_lo) st8_split(relu + pix * C + c, relu_lo + pix * C + c, o);
      else st8(relu + pix * C + c, o, false);
    }
  }
}

// ---------------------------------------------------------------- sensory GRU (modules.py:145-149, quirk Q7)
// values fp16 NHWC [B,HW,3C] = [forget | update | new]; h fp16 [B,HW,C] -> h' = f*h*(1-u) + u*tanh(n)
__global__ void __launch_bounds__(256)
gru_kernel(const __half* __restrict__ values, const __half* __restrict__ h, __half* __restrict__ out, long long pixels, int C) {
  const int C8 = C / 8;
  const long long total = pixels * C8;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long p = i / C8;
    const int c = (int)(i - p * C8) * 8;
    const __half* v = values + p * 3 * C + c;
    float f[8], u[8], n[8], hv[8], o[8];
    ld8(v, f);
    ld8(v + C, u);
    ld8(v + 2 * C, n);
    ld8(h + p * C + c, hv);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float fg = sigmoidf_(f[e]), ug = sigmoidf_(u[e]);
      o[e] = fg * hv[e] * (1.f - ug) + ug * tanhf(n[e]);
    }
    st8(out + p * C + c, o, false);
  }
}

// ---------------------------------------------------------------- key projection tail (modules.py:73-78)
// y fp32 [Q, ld] = [key(CK) | d(1) | e(CK)] -> key [Q,CK], shrinkage [Q] = d^2+1, selection [Q,CK] = sigmoid(e)
__global__ void key_tail_kernel(const float* __restrict__ y, int ld, int Q, int CK, int n_parts, long long part_stride,
                                float* __restrict__ key, float* __restrict__ shr, float* __restrict__ sel) {
  // y = n_parts fp32 partial sums (split-K of the key projection conv), added here in a fixed order with RN adds
  const long long total = (long long)Q * CK;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const long long q = i / CK;
    const int c = (int)(i - q * CK);
    const float* row = y + q * ld;
    float k = row[c], e = row[CK + 1 + c], d = (c == 0) ? row[CK] : 0.f;
    for (int p = 1; p < n_parts; ++p) {
      const float* rp = row + p * part_stride;
      k += rp[c];
      e += rp[CK + 1 + c];
      if (c == 0) d += rp[CK];
    }
    key[i] = k;
    sel[i] = sigmoidf_(e);
    if (c == 0) shr[q] = d * d + 1.f;
  }
}

// ---------------------------------------------------------------- split-K finish
// out = sum_p parts[p] (+ res + res_lo), written as fp16 (hi, lo) pairs raw and / or ReLU'd: completes a split-precision
// convolution whose K loop ran as several short accumulation chains (conv.cu, `ksplit`).  The partial sums are added
// with round-to-nearest fp32 adds in a fixed order; part 0 carries the bias.
__global__ void __launch_bounds__(256)
sum_parts_kernel(const float* __restrict__ parts, int n_parts, long long part_stride, const __half* __restrict__ res,
                 const __half* __restrict__ res_lo, __half* __restrict__ raw, __half* __restrict__ raw_lo,
                 __half* __restrict__ relu, __half* __restrict__ relu_lo, long long n8) {
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n8; i += (long long)gridDim.x * 256) {
    const long long off = i * 8;
    float v[8], t[8];
    const float4 a = *reinterpret_cast<const float4*>(parts + off), b = *reinterpret_cast<const float4*>(parts + off + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    for (int p = 1; p < n_parts; ++p) {
      const float* src = parts + p * part_stride + off;
      const float4 c = *reinterpret_cast<const float4*>(src), d = *reinterpret_cast<const float4*>(src + 4);
      v[0] += c.x; v[1] += c.y; v[2] += c.z; v[3] += c.w; v[4] += d.x; v[5] += d.y; v[6] += d.z; v[7] += d.w;
    }
    if (res) {
      ld8(res + off, t);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] += t[e];
    }
    if (res_lo) {
      ld8(res_lo + off, t);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] += t[e];
    }
    if (raw) {
      if (raw_lo) st8_split(raw + off, raw_lo + off, v);
      else st8(raw + off, v, false);
    }
    if (relu) {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = fmaxf(v[e], 0.f);
      if (relu_lo) st8_split(relu + off, relu_lo + off, v);
      else st8(relu + off, v, false);
    }
  }
}

// ---------------------------------------------------------------- output tail (network.py:33-40,144-168)
// logits fp32 [K,h,w] (pred output) -> aggregated log-odds [(K+1),h,w]
__global__ void aggregate_kernel(const float* __restrict__ logits, float* __restrict__ agg, int K, int HW) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= HW) return;
  float bg = 1.f;
  for (int k = 0; k < K; ++k) {
    const float pk = sigmoidf_(logits[(long long)k * HW + i]);
    bg *= (1.f - pk);
    const float c = fminf(fmaxf(pk, 1e-7f), 1.f - 1e-7f);
    agg[(long long)(k + 1) * HW + i] = logf(c / (1.f - c));
  }
  const float c = fminf(fmaxf(bg, 1e-7f), 1.f - 1e-7f);
  agg[i] = logf(c / (1.f - c));
}
// bilinear x4 (align_corners=False) of agg [(K+1),h,w] + softmax over channels -> prob (and logits) [(K+1),4h,4w]
__global__ void up4_softmax_kernel(const float* __restrict__ agg, float* __restrict__ prob, float* __restrict__ logits_out,
                                   int K1, int h, int w) {
  const int H = 4 * h, W = 4 * w;
  const long long i = blockIdx.x * 256ll + threadIdx.x;
  if (i >= (long long)H * W) return;
  const int Y = (int)(i / W), X = (int)(i - (long long)Y * W);
  const float sy = fmaxf((Y + 0.5f) * 0.25f - 0.5f, 0.f), sx = fmaxf((X + 0.5f) * 0.25f - 0.5f, 0.f);
  const int y0 = (int)sy, x0 = (int)sx;
  const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
  const float wy = sy - y0, wx = sx - x0;
  const long long o00 = (long long)y0 * w + x0, o01 = (long long)y0 * w + x1, o10 = (long long)y1 * w + x0,
                  o11 = (long long)y1 * w + x1;
  if (K1 <= 32) {  // the usual case: the K+1 interpolated logits stay in registers, prob is written once
    float v[32];
    float m = -CUDART_INF_F;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      if (k < K1) {
        const float* a = agg + (long long)k * h * w;
        const float top = a[o00] + (a[o01] - a[o00]) * wx, bot = a[o10] + (a[o11] - a[o10]) * wx;
        v[k] = top + (bot - top) * wy;
        if (logits_out) logits_out[(long long)k * H * W + i] = v[k];
        m = fmaxf(m, v[k]);
      }
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      if (k < K1) {
        v[k] = expf(v[k] - m);
        s += v[k];
      }
    }
    const float inv = 1.f / s;
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if (k < K1) prob[(long long)k * H * W + i] = v[k] * inv;
    return;
  }
  float m = -CUDART_INF_F;
  for (int k = 0; k < K1; ++k) {
    const float* a = agg + (long long)k * h * w;
    const float top = a[o00] + (a[o01] - a[o00]) * wx, bot = a[o10] + (a[o11] - a[o10]) * wx;
    const float v = top + (bot - top) * wy;
    prob[(long long)k * H * W + i] = v;  // stash the logit
    if (logits_out) logits_out[(long long)k * H * W + i] = v;
    m = fmaxf(m, v);
  }
  float s = 0.f;
  for (int k = 0; k < K1; ++k) {
    const float e = expf(prob[(long long)k * H * W + i] - m);
    prob[(long long)k * H * W + i] = e;
    s += e;
  }
  const float inv = 1.f / s;
  for (int k = 0; k < K1; ++k) prob[(long long)k * H * W + i] *= inv;
}

// 3x3 gather of the fused logit head: z fp32 [B,H,W,9] (z[..., t] = <relu(p4), w_t>) ->
// logits[b,y,x] = bias + sum_{t=(dy+1)*3+(dx+1)} z[b, y+dy, x+dx, t]  (zero padding)  == Conv2d(256,1,3,pad=1)
__global__ void head_gather3x3_kernel(const float* __restrict__ z, float* __restrict__ out, float bias, int B, int H, int W) {
  const long long total = (long long)B * H * W;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int x = (int)(i % W);
    long long p = i / W;
    const int y = (int)(p % H);
    const int b = (int)(p / H);
    float a = bias;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) a += z[(((long long)b * H + yy) * W + xx) * 9 + t];
    }
    out[i] = a;
  }
}

// fp16 token-major [n, C] -> fp16 bank rows dst[c, j] (ld_dst): value append from the NHWC encoder output
__global__ void transpose_append_kernel(const __half* __restrict__ src, __half* __restrict__ dst, long long ld_dst, int n,
                                        int C) {
  __shared__ __half tile[32][33];
  const int n0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int r = ty; r < 32; r += 8)
    tile[r][tx] = (n0 + r < n && c0 + tx < C) ? src[(long long)(n0 + r) * C + c0 + tx] : __float2half_rn(0.f);
  __syncthreads();
  for (int r = ty; r < 32; r += 8)
    if (c0 + r < C && n0 + tx < n) dst[(long long)(c0 + r) * ld_dst + n0 + tx] = tile[tx][r];
}
// fp32 [rows, Q] channel-major (readout GEMM output) -> fp16 NHWC-style [Q, rows]... not needed: the readout GEMM
// writes token-major directly (see readout.cu).

}  // namespace ew

static int grid_of(long long total) {
  long long g = (total + 255) / 256;
  const long long cap = (long long)sm_count() * 32;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

int ew_nchw_to_nhwc(const float* src, __half* dst, int B, int C, int H, int W, int Cp, cudaStream_t s) {
  ew::nchw_to_nhwc_kernel<<<grid_of((long long)B * H * W * Cp), 256, 0, s>>>(src, dst, B, C, H, W, Cp);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_nhwc_to_nchw(const __half* src, float* dst, int B, int C, int H, int W, cudaStream_t s) {
  ew::nhwc_to_nchw_kernel<<<grid_of((long long)B * C * H * W), 256, 0, s>>>(src, dst, B, C, H, W);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_stem_im2col(const float* src, __half* dst, __half* dst_lo, int B, int C, int H, int W, int Kp, cudaStream_t s) {
  B200_REQUIRE(H % 2 == 0 && W % 2 == 0 && Kp % 64 == 0 && Kp >= 49 * C, "stem_im2col: bad shape");
  B200_REQUIRE(C >= 1 && C <= 8, "stem_im2col: at most 8 input planes");
  const size_t smem = (size_t)C * 7 * (2 * ew::IM_XT + 5) * sizeof(float);
  // the network's shapes: one thread per output pixel, whole im2col rows written with 256-bit stores
  const dim3 gx(ceil_div(W / 2, ew::IM1_XT));
  if (C == 1 && Kp == 64 && !dst_lo) {
    ew::stem_im2col_px_kernel<1, 4, false><<<dim3(gx.x, B * ceil_div(H / 2, 4)), ew::IM1_XT, 0, s>>>(src, dst, nullptr, B, H, W);
    B200_LAUNCH_CHECK();
    return 0;
  }
  if (C == 3 && Kp == 192) {
    if (dst_lo) ew::stem_im2col_px_kernel<3, 2, true><<<dim3(gx.x, B * ceil_div(H / 2, 2)), ew::IM1_XT, 0, s>>>(src, dst, dst_lo, B, H, W);
    else ew::stem_im2col_px_kernel<3, 2, false><<<dim3(gx.x, B * ceil_div(H / 2, 2)), ew::IM1_XT, 0, s>>>(src, dst, nullptr, B, H, W);
    B200_LAUNCH_CHECK();
    return 0;
  }
  ew::stem_im2col_kernel<<<dim3(ceil_div(W / 2, ew::IM_XT), B * (H / 2)), 256, smem, s>>>(src, dst, dst_lo, B, C, H, W, Kp);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_maxpool(const __half* x, const __half* x_lo, __half* y, __half* y_lo, int B, int H, int W, int C, cudaStream_t s) {
  B200_REQUIRE(C % 8 == 0, "maxpool: C %% 8");
  ew::maxpool_kernel<<<grid_of((long long)B * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8)), 256, 0, s>>>(x, x_lo, y, y_lo, B, H, W, C);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_up2_add(const __half* g, const __half* skip, __half* raw, __half* relu, int B, int h, int w, int C, cudaStream_t s) {
  B200_REQUIRE(C % 8 == 0, "up2_add: C %% 8");
  ew::up2_add_kernel<<<dim3(ceil_div(2 * w * (C / 8), 256 * 2), B * 2 * h), 256, 0, s>>>(g, skip, raw, relu, B, h, w, C);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_up2_add_split(const __half* g, const __half* g_lo, const __half* skip, const __half* skip_lo, __half* raw,
                     __half* raw_lo, __half* relu, __half* relu_lo, unsigned char* relu_lo8, int B, int h, int w, int C,
                     cudaStream_t s) {
  B200_REQUIRE(C % 8 == 0 && g_lo && (raw != nullptr) == (raw_lo != nullptr) && (raw || relu) && (!relu_lo || relu) &&
                   (!relu_lo8 || (relu && !relu_lo)),
               "up2_add_split: C %% 8, g_lo, and raw/raw_lo (both or neither) with at least one output are required");
  ew::up2_add_split_kernel<<<dim3(ceil_div((w + 1) * (C / 8), 256), B * (h + 1)), 256, 0, s>>>(
      g, g_lo, skip, skip_lo, raw, raw_lo, relu, relu_lo, relu_lo8, B, h, w, C);
  B200_LAUNCH_CHECK();
  return 0;
}

int ew_area_down(const __half* x, __half* y, int B, int H, int W, int C, int r, cudaStream_t s) {
  B200_REQUIRE(C % 8 == 0 && H % r == 0 && W % r == 0, "area_down: shape");
  ew::area_down_kernel<<<grid_of((long long)B * (H / r) * (W / r) * (C / 8)), 256, 0, s>>>(x, y, B, H, W, C, r);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_area_down_plane(const float* x, float* y, int B, int H, int W, int r, cudaStream_t s) {
  B200_REQUIRE(H % r == 0 && W % r == 0, "area_down_plane: shape");
  ew::area_down_plane_kernel<<<grid_of((long long)B * (H / r) * (W / r)), 256, 0, s>>>(x, y, B, H, W, r);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_cbam(const __half* x, const float* w1, const float* b1, const float* w2, const float* b2, const float* ws,
            const float* bs, float* scratch, __half* raw, __half* relu, int B, int H, int W, int C, int R,
            cudaStream_t s) {
  // scratch: psum[B*16*C] | pmax[B*16*C] | gate[B*C] | stats[B*H*W*2]
  float* psum = scratch;
  float* pmax = psum + (long long)B * ew::kPoolSplit * C;
  float* gate = pmax + (long long)B * ew::kPoolSplit * C;
  float* stats = gate + (long long)B * C;
  const int HW = H * W;
  B200_REQUIRE(C % 8 == 0 && C / 8 <= 256 && 256 % (C / 8) == 0, "cbam: C = %d must be 8 x a divisor of 256", C);
  ew::cbam_pool_kernel<<<dim3(B, ew::kPoolSplit), 256, 0, s>>>(x, nullptr, psum, pmax, HW, C);
  B200_LAUNCH_CHECK();
  ew::cbam_mlp_kernel<<<B, 256, (2 * C + 2 * R) * sizeof(float), s>>>(psum, pmax, HW, w1, b1, w2, b2, gate, C, R);
  B200_LAUNCH_CHECK();
  const long long warps = (long long)B * HW;
  ew::cbam_stats_kernel<<<ceil_div(warps * 32, 256), 256, 0, s>>>(x, nullptr, gate, stats, B, HW, C);
  B200_LAUNCH_CHECK();
  ew::cbam_apply_kernel<<<ceil_div(warps * 32, 256), 256, 0, s>>>(x, gate, stats, ws, bs, raw, relu, B, H, W, C);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_cbam_split(const __half* x, const __half* x_lo, const float* w1, const float* b1, const float* w2, const float* b2,
                  const float* ws, const float* bs, float* scratch, __half* raw, __half* raw_lo, __half* relu, __half* relu_lo,
                  int pool_lo, int B, int H, int W, int C, int R, cudaStream_t s) {
  // the gate statistics are pooled over x + x_lo as well: a gate error is common to every channel of a pixel, so it
  // does not average out in the next convolution the way independent roundings do
  B200_REQUIRE(x_lo && raw && raw_lo, "cbam_split: the hi/lo tensors are required");
  float* psum = scratch;
  float* pmax = psum + (long long)B * ew::kPoolSplit * C;
  float* gate = pmax + (long long)B * ew::kPoolSplit * C;
  float* stats = gate + (long long)B * C;
  const int HW = H * W;
  B200_REQUIRE(C % 8 == 0 && C / 8 <= 256 && 256 % (C / 8) == 0, "cbam_split: C = %d must be 8 x a divisor of 256", C);
  ew::cbam_pool_kernel<<<dim3(B, ew::kPoolSplit), 256, 0, s>>>(x, pool_lo ? x_lo : nullptr, psum, pmax, HW, C);
  B200_LAUNCH_CHECK();
  ew::cbam_mlp_kernel<<<B, 256, (2 * C + 2 * R) * sizeof(float), s>>>(psum, pmax, HW, w1, b1, w2, b2, gate, C, R);
  B200_LAUNCH_CHECK();
  const long long warps = (long long)B * HW;
  ew::cbam_stats_kernel<<<ceil_div(warps * 32, 256), 256, 0, s>>>(x, pool_lo ? x_lo : nullptr, gate, stats, B, HW, C);
  B200_LAUNCH_CHECK();
  ew::cbam_apply_split_kernel<<<ceil_div(warps * 32, 256), 256, 0, s>>>(x, x_lo, gate, stats, ws, bs, raw, raw_lo, relu,
                                                                        relu_lo, B, H, W, C);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_gru(const __half* values, const __half* h, __half* out, long long pixels, int C, cudaStream_t s) {
  B200_REQUIRE(C % 8 == 0, "gru: C %% 8");
  ew::gru_kernel<<<grid_of(pixels * (C / 8)), 256, 0, s>>>(values, h, out, pixels, C);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_key_tail(const float* y, int ld, int Q, int CK, int n_parts, long long part_stride, float* key, float* shr,
                float* sel, cudaStream_t s) {
  B200_REQUIRE(n_parts >= 1, "key_tail: n_parts %d", n_parts);
  ew::key_tail_kernel<<<grid_of((long long)Q * CK), 256, 0, s>>>(y, ld, Q, CK, n_parts, part_stride, key, shr, sel);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_sum_parts(const float* parts, int n_parts, long long part_stride, const __half* res, const __half* res_lo,
                 __half* raw, __half* raw_lo, __half* relu, __half* relu_lo, long long n, cudaStream_t s) {
  B200_REQUIRE(n_parts >= 1 && n % 8 == 0 && part_stride % 4 == 0 && (raw || relu), "sum_parts: bad shape");
  ew::sum_parts_kernel<<<grid_of(n / 8), 256, 0, s>>>(parts, n_parts, part_stride, res, res_lo, raw, raw_lo, relu, relu_lo,
                                                       n / 8);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_output_tail(const float* logits, float* agg, float* prob, float* logits_out, int K, int h, int w, cudaStream_t s) {
  ew::aggregate_kernel<<<ceil_div(h * w, 256), 256, 0, s>>>(logits, agg, K, h * w);
  B200_LAUNCH_CHECK();
  ew::up4_softmax_kernel<<<ceil_div(16ll * h * w, 256), 256, 0, s>>>(agg, prob, logits_out, K + 1, h, w);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_head_gather3x3(const float* z, float* out, float bias, int B, int H, int W, cudaStream_t s) {
  ew::head_gather3x3_kernel<<<grid_of((long long)B * H * W), 256, 0, s>>>(z, out, bias, B, H, W);
  B200_LAUNCH_CHECK();
  return 0;
}
// ---------------------------------------------------------------- frame ingest / egress (SURVEY 8f-3)
namespace ew {
// u8 [h, w, 3] -> fp32 [3, h, w]: ToTensor (x / 255) then Normalize ((x - mean) / std), IEEE divisions like torch
__global__ void __launch_bounds__(256)
ingest_rgb8_kernel(const unsigned char* __restrict__ src, float* __restrict__ dst, long long hw, float m0, float m1,
                   float m2, float s0, float s1, float s2) {
  const long long i = blockIdx.x * 256ll + threadIdx.x;
  if (i >= hw) return;
  const unsigned char* p = src + 3 * i;
  dst[i] = __fdiv_rn(__fdiv_rn((float)p[0], 255.f) - m0, s0);
  dst[hw + i] = __fdiv_rn(__fdiv_rn((float)p[1], 255.f) - m1, s1);
  dst[2 * hw + i] = __fdiv_rn(__fdiv_rn((float)p[2], 255.f) - m2, s2);
}

// Source index, neighbour step (0 at the last row / column) and the two weights of output o along one axis of an
// align_corners=False bilinear resize with r = in / out: PyTorch's area_pixel_compute_source_index and
// upsample_bilinear2d_out_frame arithmetic.
__device__ __forceinline__ void bilinear_src(float r, int o, int n, int& i0, int& ip, float& l0, float& l1) {
  const float s = fmaxf(r * (o + 0.5f) - 0.5f, 0.f);
  i0 = (int)s;
  ip = i0 < n - 1 ? 1 : 0;
  l1 = s - i0;
  l0 = 1.f - l1;
}

// prob [c, h, w] -> ids [out_h, out_w]: bilinear (align_corners = False, PyTorch's upsample_bilinear2d arithmetic),
// flip, argmax (first maximum), id remap.  One thread per output pixel, channels streamed.
__global__ void __launch_bounds__(256)
prob_to_ids_kernel(const float* __restrict__ prob, int c, int h, int w, int out_h, int out_w, int flip, float rh,
                   float rw, const int* __restrict__ lut, unsigned char* __restrict__ out_u8,
                   long long* __restrict__ out_i64) {
  const long long i = blockIdx.x * 256ll + threadIdx.x;
  if (i >= (long long)out_h * out_w) return;
  const int oy = (int)(i / out_w), ox_out = (int)(i - (long long)oy * out_w);
  const int ox = flip ? out_w - 1 - ox_out : ox_out;  // flip acts on the resized map
  int best = 0;
  float best_v;
  const long long plane = (long long)h * w;
  if (out_h == h && out_w == w) {
    const float* p = prob + (long long)oy * w + ox;
    best_v = p[0];
    for (int k = 1; k < c; ++k) {
      const float v = p[k * plane];
      if (v > best_v) { best_v = v; best = k; }
    }
  } else {
    int y0, yp, x0, xp;
    float ly0, ly1, lx0, lx1;
    bilinear_src(rh, oy, h, y0, yp, ly0, ly1);
    bilinear_src(rw, ox, w, x0, xp, lx0, lx1);
    const float* p = prob + (long long)y0 * w + x0;
    best_v = -INFINITY;
    for (int k = 0; k < c; ++k) {
      const float* q = p + k * plane;
      const float v = ly0 * (lx0 * q[0] + lx1 * q[xp]) + ly1 * (lx0 * q[yp * w] + lx1 * q[yp * w + xp]);
      if (v > best_v) { best_v = v; best = k; }
    }
  }
  const int id = lut ? lut[best] : best;
  if (out_u8) out_u8[i] = (unsigned char)id;
  if (out_i64) out_i64[i] = id;
}

__device__ __forceinline__ float normalise_u8(unsigned char v, float m, float sd) {
  return __fdiv_rn(__fdiv_rn((float)v, 255.f) - m, sd);
}

// u8 [h, w, 3] -> fp32 [3, out_h, out_w]: ToTensor + Normalize per source pixel, then F.interpolate(bilinear,
// align_corners=False, antialias=False) - the demos' get_input_frame_for_deva.  One thread per output pixel.
__global__ void __launch_bounds__(256)
resize_bilinear_rgb8_kernel(const unsigned char* __restrict__ src, float* __restrict__ dst, int h, int w, int out_h,
                            int out_w, float rh, float rw, float m0, float m1, float m2, float s0, float s1, float s2) {
  const long long i = blockIdx.x * 256ll + threadIdx.x, n = (long long)out_h * out_w;
  if (i >= n) return;
  const int oy = (int)(i / out_w), ox = (int)(i - (long long)oy * out_w);
  int y0, yp, x0, xp;
  float ly0, ly1, lx0, lx1;
  bilinear_src(rh, oy, h, y0, yp, ly0, ly1);
  bilinear_src(rw, ox, w, x0, xp, lx0, lx1);
  const unsigned char* p00 = src + ((long long)y0 * w + x0) * 3;
  const unsigned char *p01 = p00 + 3 * xp, *p10 = p00 + 3ll * yp * w, *p11 = p10 + 3 * xp;
  const float m[3] = {m0, m1, m2}, sd[3] = {s0, s1, s2};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v00 = normalise_u8(p00[c], m[c], sd[c]), v01 = normalise_u8(p01[c], m[c], sd[c]);
    const float v10 = normalise_u8(p10[c], m[c], sd[c]), v11 = normalise_u8(p11[c], m[c], sd[c]);
    dst[c * n + i] = ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11);
  }
}

// Antialiased bilinear along one axis (in -> out), torch's _compute_weights_aa (aten/src/ATen/native/cpu/
// UpSampleKernel.cpp) for a float32 tensor, in its own mix of fp32 values and fp64 sums: the weights come out
// bit-identical to torch's.  Rounding scale and center to fp32 moves the taps by up to an fp32 ulp of the source
// coordinate, which is why torch's fp32 resize differs from an fp64 one by ~1e-4 on [-2.1, 2.7] data; mirroring the
// arithmetic keeps this kernel on torch's side of that gap.  Host and device share it (deva_b200_resize_aa_weights).
struct AaAxis {
  float scale, support, invscale;
  int n_in, max_taps;
};
__host__ __device__ inline AaAxis aa_axis(int n_in, int n_out) {
  AaAxis a;
  a.n_in = n_in;
  a.scale = (float)n_in / (float)n_out;
  const bool down = a.scale >= 1.f;
  a.support = down ? a.scale : 1.f;  // half the bilinear kernel width (1), stretched by scale when downscaling
  a.invscale = down ? (float)(1.0 / (double)a.scale) : 1.f;
  a.max_taps = (int)ceilf(a.support) * 2 + 1;
  return a;
}
// window [x0, x0 + n) of output i and its fp32 center
__host__ __device__ inline void aa_window(const AaAxis& a, int i, float& center, int& x0, int& n) {
  center = (float)((double)a.scale * (i + 0.5));
  const int lo = (int)((double)(center - a.support) + 0.5), hi = (int)((double)(center + a.support) + 0.5);
  x0 = lo > 0 ? lo : 0;
  n = (hi < a.n_in ? hi : a.n_in) - x0;
  n = n < 0 ? 0 : (n > a.max_taps ? a.max_taps : n);
}
// unnormalised triangle weight of source index x
__host__ __device__ inline float aa_tap(const AaAxis& a, float center, int x) {
  const float t = fabsf((float)(((double)((float)x - center) + 0.5) * (double)a.invscale));
  return t < 1.f ? 1.f - t : 0.f;
}
__host__ __device__ inline float aa_total(const AaAxis& a, float center, int x0, int n) {
  float total = 0.f;
  for (int j = 0; j < n; ++j) total += aa_tap(a, center, x0 + j);
  return total;
}
// torch leaves an all-zero window unnormalised
__host__ __device__ inline float aa_weight(const AaAxis& a, float center, int x, float total) {
  const float t = aa_tap(a, center, x);
  return total != 0.f ? t / total : t;
}

// Horizontal pass of the antialiased resize: u8 [h, w, 3] -> fp32 mid [3, h, out_w], each source pixel normalised
// (ToTensor + Normalize) before it is weighted, accumulated like torch: t = v0 * w0, then t = fma(vj, wj, t).
__global__ void __launch_bounds__(256)
resize_aa_rows_rgb8_kernel(const unsigned char* __restrict__ src, float* __restrict__ mid, int h, int w, int out_w,
                           AaAxis ax, float m0, float m1, float m2, float s0, float s1, float s2) {
  const long long i = blockIdx.x * 256ll + threadIdx.x, n_mid = (long long)h * out_w;
  if (i >= n_mid) return;
  const int y = (int)(i / out_w), ox = (int)(i - (long long)y * out_w);
  float center;
  int x0, n;
  aa_window(ax, ox, center, x0, n);
  const float total = aa_total(ax, center, x0, n);
  const unsigned char* p = src + ((long long)y * w + x0) * 3;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  for (int j = 0; j < n; ++j, p += 3) {
    const float wt = aa_weight(ax, center, x0 + j, total);
    const float v0 = normalise_u8(p[0], m0, s0), v1 = normalise_u8(p[1], m1, s1), v2 = normalise_u8(p[2], m2, s2);
    if (j == 0) {
      a0 = __fmul_rn(v0, wt); a1 = __fmul_rn(v1, wt); a2 = __fmul_rn(v2, wt);
    } else {
      a0 = __fmaf_rn(v0, wt, a0); a1 = __fmaf_rn(v1, wt, a1); a2 = __fmaf_rn(v2, wt, a2);
    }
  }
  mid[i] = a0;
  mid[n_mid + i] = a1;
  mid[2 * n_mid + i] = a2;
}

// Vertical pass: mid fp32 [3, h, out_w] -> dst [3, out_h, out_w], same accumulation.
__global__ void __launch_bounds__(256)
resize_aa_cols_kernel(const float* __restrict__ mid, float* __restrict__ dst, int h, int out_h, int out_w, AaAxis ay) {
  const long long i = blockIdx.x * 256ll + threadIdx.x, n = (long long)out_h * out_w;
  if (i >= n) return;
  const int oy = (int)(i / out_w), ox = (int)(i - (long long)oy * out_w);
  float center;
  int y0, m;
  aa_window(ay, oy, center, y0, m);
  const float total = aa_total(ay, center, y0, m);
  const long long plane = (long long)h * out_w;
  const float* p = mid + (long long)y0 * out_w + ox;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f;
  for (int j = 0; j < m; ++j, p += out_w) {
    const float wt = aa_weight(ay, center, y0 + j, total);
    if (j == 0) {
      a0 = __fmul_rn(p[0], wt); a1 = __fmul_rn(p[plane], wt); a2 = __fmul_rn(p[2 * plane], wt);
    } else {
      a0 = __fmaf_rn(p[0], wt, a0); a1 = __fmaf_rn(p[plane], wt, a1); a2 = __fmaf_rn(p[2 * plane], wt, a2);
    }
  }
  dst[i] = a0;
  dst[n + i] = a1;
  dst[2 * n + i] = a2;
}

// Palette mask u8 [h, w] -> int64 [out_h, out_w] through host-built source rows / columns (negative = outside,
// written as 0): Pillow's NEAREST resize is a pure gather once its index tables are known.
__global__ void __launch_bounds__(256)
resize_labels_kernel(const unsigned char* __restrict__ src, long long* __restrict__ dst, int w, int out_w,
                     long long n, const int* __restrict__ src_y, const int* __restrict__ src_x) {
  const long long i = blockIdx.x * 256ll + threadIdx.x;
  if (i >= n) return;
  const int oy = (int)(i / out_w), ox = (int)(i - (long long)oy * out_w);
  const int y = src_y[oy], x = src_x[ox];
  dst[i] = (y < 0 || x < 0) ? 0 : src[(long long)y * w + x];
}
}  // namespace ew

int ew_ingest_rgb8(const unsigned char* src, float* dst, int h, int w, const float* mean, const float* stdv, cudaStream_t s) {
  B200_REQUIRE(h > 0 && w > 0 && mean && stdv, "ingest_rgb8: bad arguments");
  const long long hw = (long long)h * w;
  ew::ingest_rgb8_kernel<<<(unsigned)ceil_div(hw, 256ll), 256, 0, s>>>(src, dst, hw, mean[0], mean[1], mean[2], stdv[0],
                                                                      stdv[1], stdv[2]);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_prob_to_ids(const float* prob, int c, int h, int w, int out_h, int out_w, int flip, const int* lut,
                   unsigned char* out_u8, long long* out_i64, cudaStream_t s) {
  B200_REQUIRE(c >= 1 && h > 0 && w > 0 && out_h > 0 && out_w > 0 && (out_u8 || out_i64), "prob_to_ids: bad arguments");
  const long long n = (long long)out_h * out_w;
  ew::prob_to_ids_kernel<<<(unsigned)ceil_div(n, 256ll), 256, 0, s>>>(prob, c, h, w, out_h, out_w, flip, (float)h / out_h,
                                                                     (float)w / out_w, lut, out_u8, out_i64);
  B200_LAUNCH_CHECK();
  return 0;
}
size_t ew_resize_rgb8_workspace_bytes(int h, int out_w, int mode) {
  return mode == RESIZE_READER ? sizeof(float) * 3 * (size_t)h * out_w : 0;
}
int ew_resize_rgb8(const unsigned char* src, float* dst, float* ws, int h, int w, int out_h, int out_w, int mode,
                   const float* mean, const float* stdv, cudaStream_t s) {
  B200_REQUIRE(src && dst && h > 0 && w > 0 && out_h > 0 && out_w > 0 && mean && stdv, "resize_rgb8: bad arguments");
  B200_REQUIRE(mode == RESIZE_READER || mode == RESIZE_DEMO, "resize_rgb8: unknown mode %d", mode);
  B200_REQUIRE(mode == RESIZE_DEMO || ws, "resize_rgb8: reader mode needs a workspace");
  const long long n = (long long)out_h * out_w;
  if (mode == RESIZE_DEMO) {
    ew::resize_bilinear_rgb8_kernel<<<(unsigned)ceil_div(n, 256ll), 256, 0, s>>>(
        src, dst, h, w, out_h, out_w, (float)h / out_h, (float)w / out_w, mean[0], mean[1], mean[2], stdv[0], stdv[1],
        stdv[2]);
    B200_LAUNCH_CHECK();
    return 0;
  }
  ew::resize_aa_rows_rgb8_kernel<<<(unsigned)ceil_div((long long)h * out_w, 256ll), 256, 0, s>>>(
      src, ws, h, w, out_w, ew::aa_axis(w, out_w), mean[0], mean[1], mean[2], stdv[0], stdv[1], stdv[2]);
  B200_LAUNCH_CHECK();
  ew::resize_aa_cols_kernel<<<(unsigned)ceil_div(n, 256ll), 256, 0, s>>>(ws, dst, h, out_h, out_w,
                                                                          ew::aa_axis(h, out_h));
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_resize_aa_weights(int n_in, int n_out, int max_taps, int* x0, int* n, float* wt) {
  B200_REQUIRE(n_in > 0 && n_out > 0 && max_taps > 0 && x0 && n && wt, "resize_aa_weights: bad arguments");
  const ew::AaAxis a = ew::aa_axis(n_in, n_out);
  B200_REQUIRE(a.max_taps <= max_taps, "resize_aa_weights: %d -> %d needs max_taps >= %d", n_in, n_out, a.max_taps);
  for (int i = 0; i < n_out; ++i) {
    float center;
    ew::aa_window(a, i, center, x0[i], n[i]);
    const float total = ew::aa_total(a, center, x0[i], n[i]);
    for (int j = 0; j < max_taps; ++j)
      wt[(long long)i * max_taps + j] = j < n[i] ? ew::aa_weight(a, center, x0[i] + j, total) : 0.f;
  }
  return 0;
}
int ew_resize_labels(const unsigned char* src, long long* dst, int h, int w, int out_h, int out_w, const int* src_y,
                     const int* src_x, cudaStream_t s) {
  B200_REQUIRE(src && dst && src_y && src_x && h > 0 && w > 0 && out_h > 0 && out_w > 0, "resize_labels: bad arguments");
  const long long n = (long long)out_h * out_w;
  ew::resize_labels_kernel<<<(unsigned)ceil_div(n, 256ll), 256, 0, s>>>(src, dst, w, out_w, n, src_y, src_x);
  B200_LAUNCH_CHECK();
  return 0;
}
int ew_transpose_append(const __half* src, __half* dst, long long ld_dst, int n, int C, cudaStream_t s) {
  ew::transpose_append_kernel<<<dim3(ceil_div(n, 32), ceil_div(C, 32)), 256, 0, s>>>(src, dst, ld_dst, n, C);
  B200_LAUNCH_CHECK();
  return 0;
}

}  // namespace b200
