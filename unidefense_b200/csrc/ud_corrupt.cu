// a20 -- image corruptions for corruption-robustness evaluation
//
// saturation, contrast, block, noise, blur, pixelate and baseline JPEG (4:2:0) on a batch of fp32 NCHW RGB images in
// [lo, hi], each as defined in include/unidefense_b200.h and restated in numpy by oracle/corrupt.py.  Every corruption
// works on 8-bit levels p = clamp(rint((x - lo)*s), 0, 255) and writes lo + rint(p')*(1/s), so outputs lie on the
// 8-bit grid as a decoded frame would.  saturation, contrast, block and pixelate are written as fp32 operation
// sequences with explicit rounding (__fmul_rn and friends, no FMA contraction) and are bit-identical to the oracle.
// Every output element is written by one thread from a fixed-order computation: bitwise reproducible.
//
// Launches: saturation / contrast / noise / pixelate / blur 1; block 2 (the level round trip, then the squares);
// jpeg 2 (A: one 16x16 MCU per 64 threads, colour transform + chroma subsampling + DCT -> quantise -> IDCT of the six
// blocks in shared memory, decoded planes to the workspace; B: triangle chroma upsampling, inverse colour transform).
#include <math.h>

#include <algorithm>

#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

#define CR_THREADS 256
#define CR_BLOCK_TAG 0x424C4F43u   // "BLOC"
#define CR_NOISE_TAG 0x4E4F4953u   // "NOIS"
#define CR_MAX_SIDE 8192
#define CR_BLUR_MAX_K 31

struct CrArgs {
  const float* x;
  float* y;
  const long long* ids;   // NULL: sample n has id n
  int N, H, W;
  long long HW;
  float lo, s, inv;       // p = clamp(rint((x - lo)*s), 0, 255);  y = lo + p*inv
  unsigned seed_lo, seed_hi;
};

__device__ __forceinline__ float cr_level(float x, const CrArgs& a) {
  return fminf(fmaxf(rintf(__fmul_rn(__fsub_rn(x, a.lo), a.s)), 0.f), 255.f);
}

// pre-rounding level -> output value
__device__ __forceinline__ float cr_out(float v, const CrArgs& a) {
  return __fadd_rn(a.lo, __fmul_rn(fminf(fmaxf(rintf(v), 0.f), 255.f), a.inv));
}

__device__ __forceinline__ void cr_id(const CrArgs& a, int n, unsigned& lo, unsigned& hi) {
  const unsigned long long id = a.ids ? (unsigned long long)a.ids[n] : (unsigned long long)n;
  lo = (unsigned)id;
  hi = (unsigned)(id >> 32);
}

// Philox4x32-10 (Salmon et al., SC'11), as Random123 defines it
__device__ __forceinline__ uint4 cr_philox(uint4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// Box-Muller: u1 = (a + 0.5)*2^-32, u2 = b*2^-32.  ln(u1) goes through log1p(-(1 - u1)) in the upper half, where
// 1 - u1 = (~a + 0.5)*2^-32 is exact in the integer and u1 itself would lose it to fp32 rounding.
__device__ __forceinline__ float2 cr_box_muller(unsigned a, unsigned b) {
  const float l = a < 0x80000000u ? logf(__fmul_rn(__fadd_rn((float)a, 0.5f), 0x1p-32f))
                                  : log1pf(-__fmul_rn(__fadd_rn((float)(~a), 0.5f), 0x1p-32f));
  const float r = sqrtf(-2.f * l);
  float sn, cs;
  sincospif(__fmul_rn((float)b, 0x1p-31f), &sn, &cs);
  return make_float2(r * cs, r * sn);
}

// ---- pointwise kinds: one read and one write per element ------------------------------------------------------------
#define CR_QUANT (-1)   // level round trip only (the first pass of block)

template <int KIND>
__device__ __forceinline__ void cr_pixel(const CrArgs& a, float prm, unsigned idl, unsigned idh, long long pix,
                                         float& r, float& g, float& b) {
  const float R = cr_level(r, a), G = cr_level(g, a), B = cr_level(b, a);
  if (KIND == CR_QUANT) {
    r = cr_out(R, a); g = cr_out(G, a); b = cr_out(B, a);
  } else if (KIND == UD_CORRUPT_CONTRAST) {
    r = cr_out(__fmul_rn(R, prm), a); g = cr_out(__fmul_rn(G, prm), a); b = cr_out(__fmul_rn(B, prm), a);
  } else if (KIND == UD_CORRUPT_SATURATION) {
    const float h = 128.f;
    const float Y = __fadd_rn(__fadd_rn(__fmul_rn(0.299f, R), __fmul_rn(0.587f, G)), __fmul_rn(0.114f, B));
    float Cb = __fadd_rn(__fadd_rn(__fsub_rn(__fmul_rn(-0.168736f, R), __fmul_rn(0.331264f, G)), __fmul_rn(0.5f, B)), h);
    float Cr = __fadd_rn(__fsub_rn(__fsub_rn(__fmul_rn(0.5f, R), __fmul_rn(0.418688f, G)), __fmul_rn(0.081312f, B)), h);
    Cb = __fadd_rn(h, __fmul_rn(__fsub_rn(Cb, h), prm));
    Cr = __fadd_rn(h, __fmul_rn(__fsub_rn(Cr, h), prm));
    r = cr_out(__fadd_rn(Y, __fmul_rn(1.402f, __fsub_rn(Cr, h))), a);
    g = cr_out(__fsub_rn(__fsub_rn(Y, __fmul_rn(0.344136f, __fsub_rn(Cb, h))), __fmul_rn(0.714136f, __fsub_rn(Cr, h))), a);
    b = cr_out(__fadd_rn(Y, __fmul_rn(1.772f, __fsub_rn(Cb, h))), a);
  } else {   // noise: prm = 255*sigma; chroma kept centred on 0
    const float Y = 0.299f * R + 0.587f * G + 0.114f * B;
    const float Cb = -0.168736f * R - 0.331264f * G + 0.5f * B;
    const float Cr = 0.5f * R - 0.418688f * G - 0.081312f * B;
    const uint4 w = cr_philox(make_uint4((unsigned)pix, idl, idh, 0u), a.seed_lo, a.seed_hi ^ CR_NOISE_TAG);
    const float2 z01 = cr_box_muller(w.x, w.y);
    const float z2 = cr_box_muller(w.z, w.w).x;
    const float Yn = Y + prm * z01.x, Cbn = Cb + prm * z01.y, Crn = Cr + prm * z2;
    r = cr_out(Yn + 1.402f * Crn, a);
    g = cr_out(Yn - 0.344136f * Cbn - 0.714136f * Crn, a);
    b = cr_out(Yn + 1.772f * Cbn, a);
  }
}

// VEC: 4 consecutive pixels per thread as float4 (every plane 16-byte aligned: H*W % 4 == 0 and aligned x, y)
template <int KIND, bool VEC>
__global__ void __launch_bounds__(CR_THREADS) cr_pointwise_kernel(CrArgs a, float prm) {
  const int n = blockIdx.y;
  unsigned idl, idh;
  cr_id(a, n, idl, idh);
  const long long base = (long long)n * 3 * a.HW;
  const float* x = a.x + base;
  float* y = a.y + base;
  const long long i = (long long)blockIdx.x * CR_THREADS + threadIdx.x;
  if (VEC) {
    if (4 * i >= a.HW) return;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    float4* y4 = reinterpret_cast<float4*>(y);
    const long long q = a.HW >> 2;
    float4 r = __ldg(x4 + i), g = __ldg(x4 + q + i), b = __ldg(x4 + 2 * q + i);
    cr_pixel<KIND>(a, prm, idl, idh, 4 * i + 0, r.x, g.x, b.x);
    cr_pixel<KIND>(a, prm, idl, idh, 4 * i + 1, r.y, g.y, b.y);
    cr_pixel<KIND>(a, prm, idl, idh, 4 * i + 2, r.z, g.z, b.z);
    cr_pixel<KIND>(a, prm, idl, idh, 4 * i + 3, r.w, g.w, b.w);
    y4[i] = r;
    y4[q + i] = g;
    y4[2 * q + i] = b;
  } else {
    if (i >= a.HW) return;
    float r = __ldg(x + i), g = __ldg(x + a.HW + i), b = __ldg(x + 2 * a.HW + i);
    cr_pixel<KIND>(a, prm, idl, idh, i, r, g, b);
    y[i] = r;
    y[a.HW + i] = g;
    y[2 * a.HW + i] = b;
  }
}

// ---- block: k 8x8 squares of level 128, square j from Philox(j, id) only -------------------------------------------
// Overlapping squares write the same value, so the result does not depend on which one lands last.
__global__ void __launch_bounds__(64) cr_block_kernel(CrArgs a) {
  const int j = blockIdx.x, n = blockIdx.y;
  unsigned idl, idh;
  cr_id(a, n, idl, idh);
  const uint4 u = cr_philox(make_uint4((unsigned)j, idl, idh, 0u), a.seed_lo, a.seed_hi ^ CR_BLOCK_TAG);
  const int r = (int)(((unsigned long long)u.x * (unsigned)(a.H - 7)) >> 32);
  const int c = (int)(((unsigned long long)u.y * (unsigned)(a.W - 7)) >> 32);
  const long long o = (long long)(r + (threadIdx.x >> 3)) * a.W + c + (threadIdx.x & 7);
  const float v = cr_out(128.f, a);
  float* y = a.y + (long long)n * 3 * a.HW;
  y[o] = v;
  y[a.HW + o] = v;
  y[2 * a.HW + o] = v;
}

// ---- pixelate: one CTA per (plane, f-row band); column sums of the band, then cell sums -----------------------------
// Level sums are integers <= 255*f*f, exact in fp32 in any order; the mean is one correctly rounded division.
__global__ void __launch_bounds__(CR_THREADS) cr_pixelate_kernel(CrArgs a, int f) {
  extern __shared__ float colsum[];
  const long long plane = blockIdx.x;
  const int h0 = blockIdx.y * f, rows = min(f, a.H - h0), W = a.W;
  const float* x = a.x + plane * a.HW + (long long)h0 * W;
  float* y = a.y + plane * a.HW + (long long)h0 * W;
  for (int w = threadIdx.x; w < W; w += CR_THREADS) {
    float s = 0.f;
    for (int r = 0; r < rows; ++r) s = __fadd_rn(s, cr_level(__ldg(x + (long long)r * W + w), a));
    colsum[w] = s;
  }
  __syncthreads();
  for (int w = threadIdx.x; w < W; w += CR_THREADS) {
    const int c0 = w / f * f, cols = min(f, W - c0);
    float s = 0.f;
    for (int j = 0; j < cols; ++j) s = __fadd_rn(s, colsum[c0 + j]);
    const float v = cr_out(__fdiv_rn(s, (float)(rows * cols)), a);
    for (int r = 0; r < rows; ++r) y[(long long)r * W + w] = v;
  }
}

// ---- blur: separable Gaussian on a 32x64 output tile with a reflect-101 halo in shared memory -----------------------
// Each thread filters a strip of 8 outputs from a sliding window in registers: 1 + 2R/8 shared loads per output.
struct CrBlurW {
  float w[CR_BLUR_MAX_K];
};

__device__ __forceinline__ int cr_reflect101(int i, int n) {
  i = abs(i);
  if (i >= n) i = 2 * (n - 1) - i;
  return min(max(i, 0), n - 1);   // the clamp only touches halo cells of outputs past the image edge
}

#define CR_BLUR_TW 32
#define CR_BLUR_TH 64

template <int R>
__global__ void __launch_bounds__(CR_THREADS) cr_blur_kernel(CrArgs a, CrBlurW wt, int tiles_x) {
  constexpr int TW = CR_BLUR_TW, TH = CR_BLUR_TH, IW = TW + 2 * R, IH = TH + 2 * R, K = 2 * R + 1;
  __shared__ float s_in[IH][IW];
  __shared__ float s_mid[IH][TW + 1];
  const int w0 = (blockIdx.x % tiles_x) * TW, h0 = (blockIdx.x / tiles_x) * TH;
  const long long plane = (long long)blockIdx.y * 3 + blockIdx.z;
  const float* x = a.x + plane * a.HW;
  for (int i = threadIdx.x; i < IH * IW; i += CR_THREADS) {
    const int r = i / IW, c = i - r * IW;
    const int gh = cr_reflect101(h0 - R + r, a.H), gw = cr_reflect101(w0 - R + c, a.W);
    s_in[r][c] = cr_level(__ldg(x + (long long)gh * a.W + gw), a);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < IH * (TW / 8); i += CR_THREADS) {
    const int r = i / (TW / 8), c0 = (i % (TW / 8)) * 8;
    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = 0.f;
#pragma unroll
    for (int j = 0; j < 8 + 2 * R; ++j) {
      const float v = s_in[r][c0 + j];
#pragma unroll
      for (int o = 0; o < 8; ++o)
        if (j - o >= 0 && j - o < K) acc[o] = __fmaf_rn(wt.w[j - o], v, acc[o]);
    }
#pragma unroll
    for (int o = 0; o < 8; ++o) s_mid[r][c0 + o] = acc[o];
  }
  __syncthreads();
  const int c = threadIdx.x % TW, r0 = (threadIdx.x / TW) * 8;   // 256 threads = 32 columns x 8 strips of 8 rows
  float acc[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = 0.f;
#pragma unroll
  for (int j = 0; j < 8 + 2 * R; ++j) {
    const float v = s_mid[r0 + j][c];
#pragma unroll
    for (int o = 0; o < 8; ++o)
      if (j - o >= 0 && j - o < K) acc[o] = __fmaf_rn(wt.w[j - o], v, acc[o]);
  }
  const int gw = w0 + c;
  if (gw >= a.W) return;
  float* y = a.y + plane * a.HW;
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const int gh = h0 + r0 + o;
    if (gh < a.H) y[(long long)gh * a.W + gw] = cr_out(acc[o], a);
  }
}

// ---- jpeg ----------------------------------------------------------------------------------------------------------
// The forward transform and the quantisation run in fp64, so a coefficient lands on the same side of a rounding tie
// as the fp64 definition unless it lies within ~1e-12 of the tie; the decoded planes are stored as fp32.
#define CR_MCU_PER_CTA 4

struct CrJpegQ {
  double q[128];   // luma then chroma quantisation table, natural order
};

struct CrJpegWs {
  float *Y, *Cb, *Cr;     // [N, H, W], [N, Hc, Wc] x 2
  int Hc, Wc, Mh, Mw;     // chroma plane size ceil(H/2) x ceil(W/2); MCU grid ceil(H/16) x ceil(W/16)
};

__device__ __forceinline__ double cr_rha(double v) { return copysign(floor(fabs(v) + 0.5), v); }

__global__ void __launch_bounds__(64 * CR_MCU_PER_CTA) cr_jpeg_code_kernel(CrArgs a, CrJpegWs ws, CrJpegQ Q,
                                                                          long long mcus) {
  __shared__ double s_dct[64];   // [u][m] = c(u) cos((2m+1) u pi / 16), orthonormal
  __shared__ double s_q[128];
  __shared__ double s_b[CR_MCU_PER_CTA][6][64];   // Y0 Y1 Y2 Y3 Cb Cr
  __shared__ double s_t[CR_MCU_PER_CTA][6][64];
  const int t = threadIdx.x, ty = threadIdx.y, tid = ty * 64 + t;
  if (tid < 64) s_dct[tid] = (tid < 8 ? 0.35355339059327376 : 0.5) * cospi((2 * (tid & 7) + 1) * (tid >> 3) / 16.0);
  if (tid < 128) s_q[tid] = Q.q[tid];
  const long long mcu = (long long)blockIdx.x * CR_MCU_PER_CTA + ty;
  const bool live = mcu < mcus;
  const int per = ws.Mh * ws.Mw;
  const int n = live ? (int)(mcu / per) : 0, mr = live ? (int)(mcu % per) : 0;
  const int my = mr / ws.Mw, mx = mr % ws.Mw;
  const int H = a.H, W = a.W;
  const float* x = a.x + (long long)n * 3 * a.HW;
  double* b = s_b[ty][0];
  double* tt = s_t[ty][0];
  if (live) {
    // luma, edge-replicated past the image (the padding of every plane to whole blocks)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int pix = t + 64 * j, py = pix >> 4, px = pix & 15;
      const long long o = (long long)min(16 * my + py, H - 1) * W + min(16 * mx + px, W - 1);
      const double R = cr_level(__ldg(x + o), a), G = cr_level(__ldg(x + a.HW + o), a),
                   B = cr_level(__ldg(x + 2 * a.HW + o), a);
      b[((py >> 3) * 2 + (px >> 3)) * 64 + (py & 7) * 8 + (px & 7)] = 0.299 * R + 0.587 * G + 0.114 * B - 128.0;
    }
    // chroma: 2x2 means with edge replication, the chroma plane edge-replicated to whole blocks
    const int ci = min(8 * my + (t >> 3), ws.Hc - 1), cj = min(8 * mx + (t & 7), ws.Wc - 1);
    const int rr[2] = {2 * ci, min(2 * ci + 1, H - 1)}, cc[2] = {2 * cj, min(2 * cj + 1, W - 1)};
    double cb = 0.0, cr = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long o = (long long)rr[k >> 1] * W + cc[k & 1];
      const double R = cr_level(__ldg(x + o), a), G = cr_level(__ldg(x + a.HW + o), a),
                   B = cr_level(__ldg(x + 2 * a.HW + o), a);
      cb += -0.168736 * R - 0.331264 * G + 0.5 * B + 128.0;
      cr += 0.5 * R - 0.418688 * G - 0.081312 * B + 128.0;
    }
    b[4 * 64 + t] = cb * 0.25 - 128.0;
    b[5 * 64 + t] = cr * 0.25 - 128.0;
  }
  __syncthreads();
  const int hi = t >> 3, lo = t & 7;
  // forward DCT along columns: T[u][n] = sum_m C[u][m] X[m][n]
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double s = 0.0;
#pragma unroll
    for (int m = 0; m < 8; ++m) s = fma(s_dct[hi * 8 + m], b[k * 64 + m * 8 + lo], s);
    tt[k * 64 + t] = s;
  }
  __syncthreads();
  // along rows, F[u][v] = sum_n T[u][n] C[v][n]; quantise with rha(F/Q)*Q
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double s = 0.0;
#pragma unroll
    for (int m = 0; m < 8; ++m) s = fma(tt[k * 64 + hi * 8 + m], s_dct[lo * 8 + m], s);
    const double q = s_q[(k < 4 ? 0 : 64) + t];
    b[k * 64 + t] = cr_rha(s / q) * q;
  }
  __syncthreads();
  // inverse along columns: T[m][v] = sum_u C[u][m] F[u][v]
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double s = 0.0;
#pragma unroll
    for (int u = 0; u < 8; ++u) s = fma(s_dct[u * 8 + hi], b[k * 64 + u * 8 + lo], s);
    tt[k * 64 + t] = s;
  }
  __syncthreads();
  if (!live) return;
  // along rows: X[m][n] = sum_v T[m][v] C[v][n], + 128; store the pixels inside the image
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    double s = 0.0;
#pragma unroll
    for (int v = 0; v < 8; ++v) s = fma(tt[k * 64 + hi * 8 + v], s_dct[v * 8 + lo], s);
    const float val = (float)(s + 128.0);
    if (k < 4) {
      const int gh = 16 * my + (k >> 1) * 8 + hi, gw = 16 * mx + (k & 1) * 8 + lo;
      if (gh < H && gw < W) ws.Y[(long long)n * a.HW + (long long)gh * W + gw] = val;
    } else {
      const int ci = 8 * my + hi, cj = 8 * mx + lo;
      if (ci < ws.Hc && cj < ws.Wc)
        (k == 4 ? ws.Cb : ws.Cr)[(long long)n * ws.Hc * ws.Wc + (long long)ci * ws.Wc + cj] = val;
    }
  }
}

// libjpeg's "fancy" triangle upsampling: per axis 3/4 of the nearer chroma sample + 1/4 of the next one on the
// output's side, clamped at the plane edge; rows first, then columns.
__global__ void __launch_bounds__(CR_THREADS) cr_jpeg_decode_kernel(CrArgs a, CrJpegWs ws) {
  const int n = blockIdx.y;
  const long long i = (long long)blockIdx.x * CR_THREADS + threadIdx.x;
  if (i >= a.HW) return;
  const int h = (int)(i / a.W), w = (int)(i % a.W);
  const int ni = h >> 1, fi = min(max((h & 1) ? ni + 1 : ni - 1, 0), ws.Hc - 1);
  const int nj = w >> 1, fj = min(max((w & 1) ? nj + 1 : nj - 1, 0), ws.Wc - 1);
  const long long cp = (long long)n * ws.Hc * ws.Wc;
  auto up = [&](const float* C) {
    C += cp;
    const float p = 0.75f * __ldg(C + ni * ws.Wc + nj) + 0.25f * __ldg(C + fi * ws.Wc + nj);
    const float q = 0.75f * __ldg(C + ni * ws.Wc + fj) + 0.25f * __ldg(C + fi * ws.Wc + fj);
    return 0.75f * p + 0.25f * q - 128.f;
  };
  const float Y = __ldg(ws.Y + (long long)n * a.HW + i), cb = up(ws.Cb), cr = up(ws.Cr);
  float* y = a.y + (long long)n * 3 * a.HW + i;
  y[0] = cr_out(Y + 1.402f * cr, a);
  y[a.HW] = cr_out(Y - 0.344136f * cb - 0.714136f * cr, a);
  y[2 * a.HW] = cr_out(Y + 1.772f * cb, a);
}

// ---- host ----------------------------------------------------------------------------------------------------------
static const int kCrLum[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                               14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                               18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                               49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
static const int kCrChr[16] = {17, 18, 24, 47, 18, 21, 26, 66, 24, 26, 56, 99, 47, 66, 99, 99};

// libjpeg's jpeg_quality_scaling + jpeg_add_quant_table (force_baseline)
static void cr_qtables(int q, CrJpegQ& Q) {
  const int S = q < 50 ? 5000 / q : 200 - 2 * q;
  for (int i = 0; i < 64; ++i) {
    const int r = i >> 3, c = i & 7;
    const int tc = (r < 4 && c < 4) ? kCrChr[r * 4 + c] : 99;
    Q.q[i] = (double)std::min(std::max((kCrLum[i] * S + 50) / 100, 1), 255);
    Q.q[64 + i] = (double)std::min(std::max((tc * S + 50) / 100, 1), 255);
  }
}

static bool cr_integral(float v, int lo, int hi) { return v == floorf(v) && v >= (float)lo && v <= (float)hi; }

static const char* cr_kind_name(int kind) {
  static const char* names[] = {"saturation", "contrast", "block", "noise", "blur", "pixelate", "jpeg"};
  return (kind >= 0 && kind < 7) ? names[kind] : "?";
}

extern "C" size_t ud_corrupt_workspace_bytes(int kind, int N, int H, int W) {
  if (kind != UD_CORRUPT_JPEG || N < 1 || H < 1 || W < 1) return 0;
  const size_t y = sizeof(float) * (size_t)N * H * W;
  const size_t c = sizeof(float) * (size_t)N * ((H + 1) / 2) * ((W + 1) / 2);
  return ud_align_up(y, 256) + 2 * ud_align_up(c, 256);
}

template <int KIND>
static void cr_pointwise(const CrArgs& a, float prm, bool vec, cudaStream_t stream) {
  if (vec) {
    cr_pointwise_kernel<KIND, true><<<dim3(ud_cdiv(a.HW / 4, CR_THREADS), a.N), CR_THREADS, 0, stream>>>(a, prm);
  } else {
    cr_pointwise_kernel<KIND, false><<<dim3(ud_cdiv(a.HW, CR_THREADS), a.N), CR_THREADS, 0, stream>>>(a, prm);
  }
}

template <int R>
static void cr_blur_launch(const CrArgs& a, const CrBlurW& wt, cudaStream_t stream) {
  const int tx = ud_cdiv(a.W, CR_BLUR_TW), tyy = ud_cdiv(a.H, CR_BLUR_TH);
  cr_blur_kernel<R><<<dim3(tx * tyy, a.N, 3), CR_THREADS, 0, stream>>>(a, wt, tx);
}

static void cr_blur(const CrArgs& a, int k, cudaStream_t stream) {
  const int r = (k - 1) / 2;
  const double sig = k / 6.0;
  double w[CR_BLUR_MAX_K], sum = 0.0;
  for (int i = -r; i <= r; ++i) sum += (w[i + r] = exp(-(double)i * i / (2.0 * sig * sig)));
  CrBlurW wt = {};
  for (int i = 0; i < k; ++i) wt.w[i] = (float)(w[i] / sum);
  switch (r) {
#define CR_BLUR_CASE(R_) \
  case R_: cr_blur_launch<R_>(a, wt, stream); break;
    CR_BLUR_CASE(0) CR_BLUR_CASE(1) CR_BLUR_CASE(2) CR_BLUR_CASE(3) CR_BLUR_CASE(4) CR_BLUR_CASE(5)
    CR_BLUR_CASE(6) CR_BLUR_CASE(7) CR_BLUR_CASE(8) CR_BLUR_CASE(9) CR_BLUR_CASE(10) CR_BLUR_CASE(11)
    CR_BLUR_CASE(12) CR_BLUR_CASE(13) CR_BLUR_CASE(14) CR_BLUR_CASE(15)
#undef CR_BLUR_CASE
  }
}

extern "C" int ud_corrupt(const float* x, float* y, const long long* ids, int N, int H, int W, int kind, float param,
                          unsigned long long seed, float lo, float hi, void* ws, size_t ws_bytes, cudaStream_t stream) {
  UD_REQUIRE(kind >= 0 && kind <= UD_CORRUPT_JPEG, UD_ERR_INVALID,
             "corrupt: unknown kind %d (0 saturation .. 6 jpeg)", kind);
  const char* kn = cr_kind_name(kind);
  bool ok = false;
  switch (kind) {
    case UD_CORRUPT_SATURATION:
    case UD_CORRUPT_CONTRAST: ok = param >= 0.f && param <= 1.f; break;
    case UD_CORRUPT_BLOCK: ok = cr_integral(param, 0, 4096); break;
    case UD_CORRUPT_NOISE: ok = param >= 0.f && param <= 1.f; break;
    case UD_CORRUPT_BLUR: ok = cr_integral(param, 1, CR_BLUR_MAX_K) && ((int)param & 1); break;
    case UD_CORRUPT_PIXELATE: ok = cr_integral(param, 1, 64); break;
    case UD_CORRUPT_JPEG: ok = cr_integral(param, 1, 100); break;
  }
  UD_REQUIRE(ok, UD_ERR_INVALID, "corrupt: %s parameter %g out of range", kn, (double)param);
  UD_REQUIRE(N >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "corrupt: bad shape N=%d H=%d W=%d", N, H, W);
  UD_REQUIRE(N <= 65535, UD_ERR_UNSUPPORTED, "corrupt: N=%d > 65535", N);
  UD_REQUIRE(H <= CR_MAX_SIDE && W <= CR_MAX_SIDE, UD_ERR_UNSUPPORTED, "corrupt: H=%d W=%d: sides above %d", H, W,
             CR_MAX_SIDE);
  UD_REQUIRE(kind != UD_CORRUPT_BLOCK || (H >= 8 && W >= 8), UD_ERR_INVALID,
             "corrupt: block needs H, W >= 8, got %dx%d", H, W);
  UD_REQUIRE(kind != UD_CORRUPT_BLUR || (H > ((int)param - 1) / 2 && W > ((int)param - 1) / 2), UD_ERR_INVALID,
             "corrupt: blur k=%d needs H, W > %d, got %dx%d", (int)param, ((int)param - 1) / 2, H, W);
  UD_REQUIRE(isfinite(lo) && isfinite(hi) && hi > lo, UD_ERR_INVALID, "corrupt: need hi > lo, got lo=%g hi=%g",
             (double)lo, (double)hi);
  const long long HW = (long long)H * W, total = (long long)N * 3 * HW;
  UD_REQUIRE(x && y, UD_ERR_INVALID, "corrupt: null pointer");
  UD_REQUIRE(y + total <= x || x + total <= y, UD_ERR_INVALID, "corrupt: y must not overlap x");
  const size_t need = ud_corrupt_workspace_bytes(kind, N, H, W);
  UD_REQUIRE(need == 0 || (ws && ws_bytes >= need), UD_ERR_WORKSPACE, "corrupt: workspace of %zu bytes, %zu needed",
             ws_bytes, need);

  CrArgs a;
  a.x = x; a.y = y; a.ids = ids; a.N = N; a.H = H; a.W = W; a.HW = HW;
  const double s = 255.0 / ((double)hi - (double)lo);
  a.lo = lo; a.s = (float)s; a.inv = (float)(1.0 / s);
  a.seed_lo = (unsigned)seed;
  a.seed_hi = (unsigned)(seed >> 32);
  const bool vec = HW % 4 == 0 && (((uintptr_t)x | (uintptr_t)y) & 15) == 0;

  switch (kind) {
    case UD_CORRUPT_SATURATION: cr_pointwise<UD_CORRUPT_SATURATION>(a, param, vec, stream); break;
    case UD_CORRUPT_CONTRAST: cr_pointwise<UD_CORRUPT_CONTRAST>(a, param, vec, stream); break;
    case UD_CORRUPT_NOISE: cr_pointwise<UD_CORRUPT_NOISE>(a, (float)(255.0 * sqrt((double)param)), vec, stream); break;
    case UD_CORRUPT_BLOCK: {
      cr_pointwise<CR_QUANT>(a, 0.f, vec, stream);
      const int k = (int)param;
      if (k > 0) {
        const int rc = ud_check_launch("corrupt (block levels)");
        if (rc) return rc;
        cr_block_kernel<<<dim3(k, N), 64, 0, stream>>>(a);
      }
      break;
    }
    case UD_CORRUPT_BLUR: cr_blur(a, (int)param, stream); break;
    case UD_CORRUPT_PIXELATE: {
      const int f = (int)param;
      cr_pixelate_kernel<<<dim3(3 * N, ud_cdiv(H, f)), CR_THREADS, sizeof(float) * W, stream>>>(a, f);
      break;
    }
    case UD_CORRUPT_JPEG: {
      CrJpegQ Q;
      cr_qtables((int)param, Q);
      CrJpegWs w;
      w.Hc = (H + 1) / 2; w.Wc = (W + 1) / 2; w.Mh = (H + 15) / 16; w.Mw = (W + 15) / 16;
      char* p = (char*)ws;
      w.Y = (float*)p;
      p += ud_align_up(sizeof(float) * (size_t)N * HW, 256);
      w.Cb = (float*)p;
      w.Cr = (float*)(p + ud_align_up(sizeof(float) * (size_t)N * w.Hc * w.Wc, 256));
      const long long mcus = (long long)N * w.Mh * w.Mw;
      cr_jpeg_code_kernel<<<ud_cdiv(mcus, CR_MCU_PER_CTA), dim3(64, CR_MCU_PER_CTA), 0, stream>>>(a, w, Q, mcus);
      const int rc = ud_check_launch("corrupt (jpeg code)");
      if (rc) return rc;
      cr_jpeg_decode_kernel<<<dim3(ud_cdiv(HW, CR_THREADS), N), CR_THREADS, 0, stream>>>(a, w);
      break;
    }
  }
  return ud_check_launch("corrupt");
}
