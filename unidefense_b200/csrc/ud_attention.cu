// a4 / a7 -- attention() glue: bilinear resize, error maps, feature-map rFFT2 / irFFT2 and the
// sigmoid-gated fuse                                            (SURVEY.md §8a rows a4, a7)
//
// Reference: model/unidefense.py:125-157 (Eb4), :329-361 (Res18), :522-554 (Res50).
// Feature maps on this path are small (12x12, 8x8, 16x16, 24x24 ...; SURVEY App. A.1), so one
// plane lives entirely in shared memory and the 2-D transform is evaluated as two passes of
// direct DFTs against sincospif-exact twiddle tables: HBM traffic is one read + one write.
// Spectra use the reference's channel-planar cat([re, im], dim=1) layout.
#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

#define AT_THREADS 256
#define AT_MAX_DIM 64   // small-plane path: h, w <= 64

// ---------------------------------------------------------------- bilinear resize (align_corners)
__global__ void at_bilinear_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long total, int h,
                                       int w, int H, int W, float sy, float sx) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % W);
    const long long t = i / W;
    const int r = (int)(t % H);
    const long long plane = t / H;
    const UdLerp yr = ud_lerp_ac(r, h, sy), xc = ud_lerp_ac(c, w, sx);
    const float* p = x + plane * (long long)h * w;
    y[i] = yr.l0 * (xc.l0 * __ldg(p + yr.i0 * w + xc.i0) + xc.l1 * __ldg(p + yr.i0 * w + xc.i1)) +
           yr.l1 * (xc.l0 * __ldg(p + yr.i1 * w + xc.i0) + xc.l1 * __ldg(p + yr.i1 * w + xc.i1));
  }
}
// transposed resize (upsample_bilinear2d_backward): gx pre-zeroed, scatter with atomics
__global__ void at_bilinear_bwd_kernel(const float* __restrict__ gy, float* __restrict__ gx, long long total, int h,
                                       int w, int H, int W, float sy, float sx) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % W);
    const long long t = i / W;
    const int r = (int)(t % H);
    const long long plane = t / H;
    const UdLerp yr = ud_lerp_ac(r, h, sy), xc = ud_lerp_ac(c, w, sx);
    float* p = gx + plane * (long long)h * w;
    const float g = gy[i];
    atomicAdd(p + yr.i0 * w + xc.i0, yr.l0 * xc.l0 * g);
    atomicAdd(p + yr.i0 * w + xc.i1, yr.l0 * xc.l1 * g);
    atomicAdd(p + yr.i1 * w + xc.i0, yr.l1 * xc.l0 * g);
    atomicAdd(p + yr.i1 * w + xc.i1, yr.l1 * xc.l1 * g);
  }
}

extern "C" int ud_bilinear_ac_fwd(const float* x, float* y, int planes, int h, int w, int H, int W,
                                  cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && h >= 1 && w >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "bilinear_fwd: bad shape");
  const long long total = (long long)planes * H * W;
  if (total == 0) return UD_OK;
  UD_REQUIRE(x && y, UD_ERR_INVALID, "bilinear_fwd: null pointer");
  const int blocks = (int)min((long long)UD_NUM_SMS * 8, (total + 255) / 256);
  at_bilinear_fwd_kernel<<<blocks, 256, 0, stream>>>(x, y, total, h, w, H, W, ud_ac_scale(h, H), ud_ac_scale(w, W));
  return ud_check_launch("bilinear_fwd");
}
extern "C" int ud_bilinear_ac_bwd(const float* gy, float* gx, int planes, int h, int w, int H, int W,
                                  cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && h >= 1 && w >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "bilinear_bwd: bad shape");
  const long long total = (long long)planes * H * W;
  if ((long long)planes * h * w == 0) return UD_OK;
  UD_REQUIRE(gy && gx, UD_ERR_INVALID, "bilinear_bwd: null pointer");
  UD_CUDA(cudaMemsetAsync(gx, 0, sizeof(float) * (size_t)planes * h * w, stream));
  const int blocks = (int)min((long long)UD_NUM_SMS * 8, (total + 255) / 256);
  at_bilinear_bwd_kernel<<<blocks, 256, 0, stream>>>(gy, gx, total, h, w, H, W, ud_ac_scale(h, H), ud_ac_scale(w, W));
  return ud_check_launch("bilinear_bwd");
}

// ---------------------------------------------------------------- small-plane 2-D DFTs
// twiddle tables e^{-2 pi i t/n} as (cos, -sin)
__device__ __forceinline__ void at_fill_tw(float2* tw, int n, int tid, int nthreads) {
  for (int t = tid; t < n; t += nthreads) {
    float s, c;
    sincospif(2.0f * (float)t / (float)n, &s, &c);
    tw[t] = make_float2(c, -s);
  }
}

// Real -> half spectrum for one plane held in shared memory.
//   src [h][w] real (smem), tmp [h][wh] complex (smem), twW [w], twH [h].
//   emits X[j][k] * scale * (colmul ? m_k : 1) through `emit(j, k, re, im)`.
template <class Emit>
__device__ __forceinline__ void at_r2c_plane(const float* src, float2* tmp, const float2* twW, const float2* twH, int h,
                                             int w, float scale, bool colmul, int lt, int tpp, Emit emit) {
  const int wh = w / 2 + 1;
  for (int o = lt; o < h * wh; o += tpp) {
    const int r = o / wh, k = o - r * wh;
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int c = 0; c < w; ++c) {
      const float v = src[r * w + c];
      const float2 t = twW[idx];
      re = fmaf(v, t.x, re);
      im = fmaf(v, t.y, im);
      idx += k;
      if (idx >= w) idx -= w;
    }
    tmp[o] = make_float2(re, im);
  }
  __syncthreads();
  const int last = (w % 2 == 0) ? wh - 1 : wh;
  for (int o = lt; o < h * wh; o += tpp) {
    const int j = o / wh, k = o - j * wh;
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int r = 0; r < h; ++r) {
      const float2 v = tmp[r * wh + k];
      const float2 t = twH[idx];
      re += v.x * t.x - v.y * t.y;
      im += v.x * t.y + v.y * t.x;
      idx += j;
      if (idx >= h) idx -= h;
    }
    const float m = (colmul && k >= 1 && k < last) ? 2.f * scale : scale;
    emit(j, k, re * m, im * m);
  }
}

// Half spectrum -> real for one plane:  y[r][c] = scale * sum_k m_k Re(U[r][k] e^{+2 pi i k c/w}),
// U[r][k] = sum_j Z[j][k] e^{+2 pi i j r/h};  m_k = 1 when !colmul (plain adjoint of r2c).
//   spec [h][wh] complex (smem), tmp [h][wh] complex (smem)
template <class Emit>
__device__ __forceinline__ void at_c2r_plane(const float2* spec, float2* tmp, const float2* twW, const float2* twH,
                                             int h, int w, float scale, bool colmul, int lt, int tpp, Emit emit) {
  const int wh = w / 2 + 1;
  for (int o = lt; o < h * wh; o += tpp) {
    const int r = o / wh, k = o - r * wh;
    float re = 0.f, im = 0.f;
    int idx = 0;
    for (int j = 0; j < h; ++j) {
      const float2 v = spec[j * wh + k];
      const float2 t = twH[idx];  // (cos, -sin): conj for the inverse
      re += v.x * t.x + v.y * t.y;
      im += v.y * t.x - v.x * t.y;
      idx += r;
      if (idx >= h) idx -= h;
    }
    tmp[o] = make_float2(re, im);
  }
  __syncthreads();
  const int last = (w % 2 == 0) ? wh - 1 : wh;
  for (int o = lt; o < h * w; o += tpp) {
    const int r = o / w, c = o - r * w;
    float acc = 0.f;
    int idx = 0;
    for (int k = 0; k < wh; ++k) {
      const float2 v = tmp[r * wh + k];
      const float2 t = twW[idx];
      // Re(v * (cos + i sin)) = v.x cos - v.y sin = v.x*t.x + v.y*t.y
      const float term = v.x * t.x + v.y * t.y;
      acc += (colmul && k >= 1 && k < last) ? 2.f * term : term;
      idx += c;
      if (idx >= w) idx -= w;
    }
    emit(r, c, acc * scale);
  }
}

// floats per plane slot: real plane padded to an even count (keeps the float2 regions 8-byte
// aligned) + two complex half-spectrum buffers
__host__ __device__ static inline int at_slot_floats(int h, int w) {
  const int wh = w / 2 + 1;
  return ((h * w + 1) & ~1) + 4 * h * wh;
}
static inline int at_planes_per_cta(int h, int w) {
  const size_t per = sizeof(float) * (size_t)at_slot_floats(h, w);
  int p = (int)((40u << 10) / per);
  if (p < 1) p = 1;
  if (p > 8) p = 8;
  while (AT_THREADS % p) --p;
  return p;
}
static inline size_t at_smem_bytes(int h, int w, int P) {
  return sizeof(float2) * (size_t)(w + h) + (size_t)P * sizeof(float) * (size_t)at_slot_floats(h, w);
}

// x [N,C,h,w] -> out [N,2C,h,wh]  (cat_rfft2; also irfft2 backward with colmul)
__global__ void __launch_bounds__(AT_THREADS)
at_r2c_kernel(const float* __restrict__ x, float* __restrict__ out, int planes, int C, int h, int w, float scale,
              int colmul, int P) {
  extern __shared__ float2 sm2[];
  const int wh = w / 2 + 1;
  float2* twW = sm2;
  float2* twH = twW + w;
  float* base = reinterpret_cast<float*>(twH + h);
  const int tpp = AT_THREADS / P;
  const int lp = threadIdx.x / tpp, lt = threadIdx.x - lp * tpp;
  float* src = base + (size_t)lp * at_slot_floats(h, w);
  float2* tmp = reinterpret_cast<float2*>(src + ((h * w + 1) & ~1));
  at_fill_tw(twW, w, threadIdx.x, AT_THREADS);
  at_fill_tw(twH, h, threadIdx.x, AT_THREADS);
  const int plane = blockIdx.x * P + lp;
  const bool live = plane < planes;
  if (live) {
    const float* xp = x + (long long)plane * h * w;
    for (int i = lt; i < h * w; i += tpp) src[i] = xp[i];
  } else {
    for (int i = lt; i < h * w; i += tpp) src[i] = 0.f;
  }
  __syncthreads();
  const int n = live ? plane / C : 0, c = live ? plane % C : 0;
  float* ore = out + ((long long)n * 2 * C + c) * h * wh;
  float* oim = out + ((long long)n * 2 * C + C + c) * h * wh;
  at_r2c_plane(src, tmp, twW, twH, h, w, scale, colmul != 0, lt, tpp, [&](int j, int k, float re, float im) {
    if (live) {
      ore[j * wh + k] = re;
      oim[j * wh + k] = im;
    }
  });
}

// in [N,2C,h,wh] (optionally multiplied by mask [N,h*wh]) -> y [N,C,h,w]   (irfft2_from_cat; also rfft2 backward)
__global__ void __launch_bounds__(AT_THREADS)
at_c2r_kernel(const float* __restrict__ in, const float* __restrict__ mask, float* __restrict__ y, int planes, int C,
              int h, int w, float scale, int colmul, int P) {
  extern __shared__ float2 sm2[];
  const int wh = w / 2 + 1;
  float2* twW = sm2;
  float2* twH = twW + w;
  float* base = reinterpret_cast<float*>(twH + h);
  const int tpp = AT_THREADS / P;
  const int lp = threadIdx.x / tpp, lt = threadIdx.x - lp * tpp;
  float* reg = base + (size_t)lp * at_slot_floats(h, w);
  float2* spec = reinterpret_cast<float2*>(reg + ((h * w + 1) & ~1));
  float2* tmp = spec + h * wh;
  at_fill_tw(twW, w, threadIdx.x, AT_THREADS);
  at_fill_tw(twH, h, threadIdx.x, AT_THREADS);
  const int plane = blockIdx.x * P + lp;
  const bool live = plane < planes;
  const int n = live ? plane / C : 0, c = live ? plane % C : 0;
  if (live) {
    const float* ire = in + ((long long)n * 2 * C + c) * h * wh;
    const float* iim = in + ((long long)n * 2 * C + C + c) * h * wh;
    const float* mk = mask ? mask + (long long)n * h * wh : nullptr;
    for (int i = lt; i < h * wh; i += tpp) {
      const float m = mk ? mk[i] : 1.f;
      spec[i] = make_float2(ire[i] * m, iim[i] * m);
    }
  } else {
    for (int i = lt; i < h * wh; i += tpp) spec[i] = make_float2(0.f, 0.f);
  }
  __syncthreads();
  float* yp = y + (long long)plane * h * w;
  at_c2r_plane(spec, tmp, twW, twH, h, w, scale, colmul != 0, lt, tpp, [&](int r, int cc, float v) {
    if (live) yp[r * w + cc] = v;
  });
}

static int at_check_small(const char* what, int N, int C, int h, int w) {
  UD_REQUIRE(N >= 0 && C >= 1 && h >= 1 && w >= 1, UD_ERR_INVALID, "%s: bad shape N=%d C=%d h=%d w=%d", what, N, C, h, w);
  UD_REQUIRE(h <= AT_MAX_DIM && w <= AT_MAX_DIM, UD_ERR_UNSUPPORTED,
             "%s: plane %dx%d exceeds the small-plane path (max %d); use ud_rfft2 / ud_irfft2", what, h, w, AT_MAX_DIM);
  return UD_OK;
}

template <class K>
static int at_set_smem(K k, size_t bytes) {
  if (bytes > (48u << 10)) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      ud_set_error("cudaFuncSetAttribute(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return UD_ERR_CUDA;
    }
  }
  return UD_OK;
}

static float at_scale(int h, int w, int norm_ortho, bool inverse) {
  if (norm_ortho) return 1.f / sqrtf((float)h * (float)w);
  return inverse ? 1.f / ((float)h * (float)w) : 1.f;
}

// mode 0: forward transform (scale per norm);  mode 1: adjoint of the inverse transform (irfft2 backward)
bool ud_fft2_small_ok(int h, int w) { return h <= AT_MAX_DIM && w <= AT_MAX_DIM; }

int ud_rfft2_small(const float* x, float* xf, int N, int C, int h, int w, int norm_ortho, int adjoint_of_inverse,
                   cudaStream_t stream) {
  int rc;
  const int P = at_planes_per_cta(h, w);
  const size_t smem = at_smem_bytes(h, w, P);
  if ((rc = at_set_smem(at_r2c_kernel, smem)) != UD_OK) return rc;
  const int planes = N * C;
  const float scale = at_scale(h, w, norm_ortho, adjoint_of_inverse != 0);
  at_r2c_kernel<<<ud_cdiv(planes, P), AT_THREADS, smem, stream>>>(x, xf, planes, C, h, w, scale, adjoint_of_inverse, P);
  return ud_check_launch("rfft2_cat");
}

// mode 0: inverse transform irfft2(s=(h,w)) (column multipliers m_k, scale per norm);
// mode 1: adjoint of the forward transform (rfft2 backward: zero-padded, no multipliers)
int ud_irfft2_small(const float* xf, const float* mask, float* y, int N, int C, int h, int w, int norm_ortho,
                    int adjoint_of_forward, cudaStream_t stream) {
  int rc;
  const int P = at_planes_per_cta(h, w);
  const size_t smem = at_smem_bytes(h, w, P);
  if ((rc = at_set_smem(at_c2r_kernel, smem)) != UD_OK) return rc;
  const int planes = N * C;
  const float scale = at_scale(h, w, norm_ortho, adjoint_of_forward == 0);
  at_c2r_kernel<<<ud_cdiv(planes, P), AT_THREADS, smem, stream>>>(xf, mask, y, planes, C, h, w, scale,
                                                                   adjoint_of_forward ? 0 : 1, P);
  return ud_check_launch("irfft2_cat");
}

// ---------------------------------------------------------------- a4: error maps
// d = down(pred) - down(x) at small-plane pixel (r, cc) for the backward: the expression of at_prep_kernel below, so
// that the backward sees the forward's fp32 value (and so its signs)
__device__ __forceinline__ float at_prep_d(const float* __restrict__ pp, const float* __restrict__ xp, int r, int cc,
                                           int hp, int wp, int Hx, int Wx, float syp, float sxp, float syx, float sxx) {
  UdLerp yr = ud_lerp_ac(r, hp, syp), xc = ud_lerp_ac(cc, wp, sxp);
  const float pv = yr.l0 * (xc.l0 * __ldg(pp + yr.i0 * wp + xc.i0) + xc.l1 * __ldg(pp + yr.i0 * wp + xc.i1)) +
                   yr.l1 * (xc.l0 * __ldg(pp + yr.i1 * wp + xc.i0) + xc.l1 * __ldg(pp + yr.i1 * wp + xc.i1));
  yr = ud_lerp_ac(r, Hx, syx);
  xc = ud_lerp_ac(cc, Wx, sxx);
  const float xv = yr.l0 * (xc.l0 * __ldg(xp + (long long)yr.i0 * Wx + xc.i0) + xc.l1 * __ldg(xp + (long long)yr.i0 * Wx + xc.i1)) +
                   yr.l1 * (xc.l0 * __ldg(xp + (long long)yr.i1 * Wx + xc.i0) + xc.l1 * __ldg(xp + (long long)yr.i1 * Wx + xc.i1));
  return pv - xv;
}

// pred [N,C,hp,wp], x [N,C,Hx,Wx] -> spat_diff [N,C,h,w] = |p - xs|, freq_diff [N,2C,h,wh] = |cat rfft2(p - xs)|
// (model/unidefense.py:126-134,:148; one FFT by linearity).  One CTA per (n,c) plane.
__global__ void __launch_bounds__(AT_THREADS)
at_prep_kernel(const float* __restrict__ pred, const float* __restrict__ x, float* __restrict__ spat_diff,
               float* __restrict__ freq_diff, int C, int hp, int wp, int Hx, int Wx, int h, int w, float syp,
               float sxp, float syx, float sxx, float scale) {
  extern __shared__ float2 sm2[];
  const int wh = w / 2 + 1;
  float2* twW = sm2;
  float2* twH = twW + w;
  float* src = reinterpret_cast<float*>(twH + h);
  float2* tmp = reinterpret_cast<float2*>(src + ((h * w + 1) & ~1));
  at_fill_tw(twW, w, threadIdx.x, AT_THREADS);
  at_fill_tw(twH, h, threadIdx.x, AT_THREADS);
  const int plane = blockIdx.x;
  const int n = plane / C, c = plane % C;
  const float* pp = pred + (long long)plane * hp * wp;
  const float* xp = x + (long long)plane * Hx * Wx;
  float* sd = spat_diff + (long long)plane * h * w;
  for (int i = threadIdx.x; i < h * w; i += AT_THREADS) {
    const int r = i / w, cc = i - r * w;
    UdLerp yr = ud_lerp_ac(r, hp, syp), xc = ud_lerp_ac(cc, wp, sxp);
    const float pv = yr.l0 * (xc.l0 * __ldg(pp + yr.i0 * wp + xc.i0) + xc.l1 * __ldg(pp + yr.i0 * wp + xc.i1)) +
                     yr.l1 * (xc.l0 * __ldg(pp + yr.i1 * wp + xc.i0) + xc.l1 * __ldg(pp + yr.i1 * wp + xc.i1));
    yr = ud_lerp_ac(r, Hx, syx);
    xc = ud_lerp_ac(cc, Wx, sxx);
    const float xv = yr.l0 * (xc.l0 * __ldg(xp + (long long)yr.i0 * Wx + xc.i0) + xc.l1 * __ldg(xp + (long long)yr.i0 * Wx + xc.i1)) +
                     yr.l1 * (xc.l0 * __ldg(xp + (long long)yr.i1 * Wx + xc.i0) + xc.l1 * __ldg(xp + (long long)yr.i1 * Wx + xc.i1));
    const float d = pv - xv;
    src[i] = d;
    sd[i] = fabsf(d);
  }
  __syncthreads();
  float* ore = freq_diff + ((long long)n * 2 * C + c) * h * wh;
  float* oim = freq_diff + ((long long)n * 2 * C + C + c) * h * wh;
  at_r2c_plane(src, tmp, twW, twH, h, w, scale, false, threadIdx.x, AT_THREADS, [&](int j, int k, float re, float im) {
    ore[j * wh + k] = fabsf(re);
    oim[j * wh + k] = fabsf(im);
  });
}

extern "C" int ud_attn_prep(const float* pred, const float* x, float* spat_diff, float* freq_diff, int N, int C, int hp,
                            int wp, int Hx, int Wx, int h, int w, int norm_ortho, cudaStream_t stream) {
  int rc = at_check_small("attn_prep", N, C, h, w);
  if (rc != UD_OK) return rc;
  UD_REQUIRE(hp >= 1 && wp >= 1 && Hx >= 1 && Wx >= 1, UD_ERR_INVALID, "attn_prep: bad source shape");
  if (N == 0) return UD_OK;
  UD_REQUIRE(pred && x && spat_diff && freq_diff, UD_ERR_INVALID, "attn_prep: null pointer");
  const size_t smem = at_smem_bytes(h, w, 1);
  if ((rc = at_set_smem(at_prep_kernel, smem)) != UD_OK) return rc;
  at_prep_kernel<<<N * C, AT_THREADS, smem, stream>>>(pred, x, spat_diff, freq_diff, C, hp, wp, Hx, Wx, h, w,
                                                      ud_ac_scale(hp, h), ud_ac_scale(wp, w), ud_ac_scale(Hx, h),
                                                      ud_ac_scale(Wx, w), at_scale(h, w, norm_ortho, false));
  return ud_check_launch("attn_prep");
}

// ---------------------------------------------------------------- a4 backward: error maps -> x
// g_d = sign(d) * g_sd + fft_r2c_backward(sign(F) * g_fd) at (h, w); g_x = -(transposed align-corners resize)(g_d).
// grid (row tiles of the x plane, N*C planes).  Every CTA recomputes d and the small-plane transforms of its plane
// (<= 64x64, the same code and thread mapping as at_prep_kernel, so the signs are the forward's), then GATHERS its
// rows of g_x: output pixel (R, Q) reads the small pixels whose bilinear taps include it, in a fixed order.  g_x is
// written once, coalesced, without atomics: bitwise reproducible.
#define AT_BWD_ROWS 8   // x rows per CTA

// small-plane index range [lo, hi] whose align-corners taps (scale s = (in-1)/(out-1), in = big, out = small) can
// include big index R; the weights are then evaluated exactly with ud_lerp_ac
__device__ __forceinline__ void at_tap_range(int R, int out, float s, int& lo, int& hi) {
  if (s <= 0.f) {                     // out == 1 (s = 0): every small index samples big index 0
    lo = 0;
    hi = out - 1;
    return;
  }
  lo = max(0, (int)floorf((float)(R - 1) / s) - 1);
  hi = min(out - 1, (int)ceilf((float)(R + 1) / s) + 1);
}
__device__ __forceinline__ float at_tap_weight(int r, int R, int in, float s) {
  const UdLerp l = ud_lerp_ac(r, in, s);
  return (l.i0 == R ? l.l0 : 0.f) + (l.i1 == R ? l.l1 : 0.f);
}

__global__ void __launch_bounds__(AT_THREADS)
at_prep_bwd_kernel(const float* __restrict__ pred, const float* __restrict__ x, const float* __restrict__ g_sd,
                   const float* __restrict__ g_fd, float* __restrict__ g_x, int C, int hp, int wp, int Hx, int Wx, int h,
                   int w, float syp, float sxp, float syx, float sxx, float scale) {
  extern __shared__ float2 sm2[];
  const int wh = w / 2 + 1;
  float2* twW = sm2;
  float2* twH = twW + w;
  float* gd = reinterpret_cast<float*>(twH + h);               // d, then g_d [h][w]
  float2* tmp = reinterpret_cast<float2*>(gd + ((h * w + 1) & ~1));
  float2* spec = tmp + h * wh;
  at_fill_tw(twW, w, threadIdx.x, AT_THREADS);
  at_fill_tw(twH, h, threadIdx.x, AT_THREADS);
  const int plane = blockIdx.y;
  const int n = plane / C, c = plane % C;
  const float* pp = pred + (long long)plane * hp * wp;
  const float* xp = x + (long long)plane * Hx * Wx;
  for (int i = threadIdx.x; i < h * w; i += AT_THREADS) {
    const int r = i / w, cc = i - r * w;
    gd[i] = at_prep_d(pp, xp, r, cc, hp, wp, Hx, Wx, syp, sxp, syx, sxx);
  }
  __syncthreads();
  const float* gsp = g_sd ? g_sd + (long long)plane * h * w : nullptr;
  if (g_fd != nullptr) {
    const float* gre = g_fd + ((long long)n * 2 * C + c) * h * wh;
    const float* gim = g_fd + ((long long)n * 2 * C + C + c) * h * wh;
    at_r2c_plane(gd, tmp, twW, twH, h, w, scale, false, threadIdx.x, AT_THREADS, [&](int j, int k, float re, float im) {
      const int o = j * wh + k;
      spec[o] = make_float2(ud_sign(re) * __ldg(gre + o), ud_sign(im) * __ldg(gim + o));
    });
    __syncthreads();                  // tmp is reused by the inverse
    at_c2r_plane(spec, tmp, twW, twH, h, w, scale, false, threadIdx.x, AT_THREADS, [&](int r, int cc, float v) {
      const int i = r * w + cc;
      gd[i] = gsp ? fmaf(ud_sign(gd[i]), __ldg(gsp + i), v) : v;
    });
  } else {
    for (int i = threadIdx.x; i < h * w; i += AT_THREADS) gd[i] = gsp ? ud_sign(gd[i]) * __ldg(gsp + i) : 0.f;
  }
  __syncthreads();
  float* gxp = g_x + (long long)plane * Hx * Wx;
  const int R0 = blockIdx.x * AT_BWD_ROWS, R1 = min(Hx, R0 + AT_BWD_ROWS);
  for (int Q = threadIdx.x; Q < Wx; Q += AT_THREADS) {
    int clo, chi;
    at_tap_range(Q, w, sxx, clo, chi);
    for (int R = R0; R < R1; ++R) {
      int rlo, rhi;
      at_tap_range(R, h, syx, rlo, rhi);
      float acc = 0.f;
      for (int r = rlo; r <= rhi; ++r) {
        const float wr = at_tap_weight(r, R, Hx, syx);
        if (wr == 0.f) continue;
        float row = 0.f;
        for (int cc = clo; cc <= chi; ++cc) {
          const float wc = at_tap_weight(cc, Q, Wx, sxx);
          if (wc != 0.f) row = fmaf(wc, gd[r * w + cc], row);
        }
        acc = fmaf(wr, row, acc);
      }
      gxp[(long long)R * Wx + Q] = -acc;
    }
  }
}

extern "C" int ud_attn_prep_bwd(const float* pred, const float* x, const float* g_spat_diff, const float* g_freq_diff,
                                float* g_x, int N, int C, int hp, int wp, int Hx, int Wx, int h, int w, int norm_ortho,
                                cudaStream_t stream) {
  int rc = at_check_small("attn_prep_bwd", N, C, h, w);
  if (rc != UD_OK) return rc;
  UD_REQUIRE(hp >= 1 && wp >= 1 && Hx >= 1 && Wx >= 1, UD_ERR_INVALID, "attn_prep_bwd: bad source shape");
  UD_REQUIRE((long long)N * C <= 65535, UD_ERR_UNSUPPORTED, "attn_prep_bwd: too many planes (%lld)", (long long)N * C);
  if (N == 0) return UD_OK;
  UD_REQUIRE(pred && x && g_x, UD_ERR_INVALID, "attn_prep_bwd: null pointer");
  const size_t smem = sizeof(float2) * (size_t)(w + h) + sizeof(float) * (size_t)at_slot_floats(h, w);
  if ((rc = at_set_smem(at_prep_bwd_kernel, smem)) != UD_OK) return rc;
  at_prep_bwd_kernel<<<dim3(ud_cdiv(Hx, AT_BWD_ROWS), N * C), AT_THREADS, smem, stream>>>(
      pred, x, g_spat_diff, g_freq_diff, g_x, C, hp, wp, Hx, Wx, h, w, ud_ac_scale(hp, h), ud_ac_scale(wp, w),
      ud_ac_scale(Hx, h), ud_ac_scale(Wx, w), at_scale(h, w, norm_ortho, false));
  return ud_check_launch("attn_prep_bwd");
}

// ---------------------------------------------------------------- a7: fuse
// out = (1-s)*smask*emb + s*ff + res,  s = sigmoid(*fuse_coef)   (model/unidefense.py:153-155)
//   emb, ff, res [N,C,HW]; smask [N,HW]; res = dropout(emb.clone()) (nullable -> emb)
__global__ void at_fuse_fwd_kernel(const float* __restrict__ emb, const float* __restrict__ smask,
                                   const float* __restrict__ ff, const float* __restrict__ res,
                                   const float* __restrict__ fuse_coef, float* __restrict__ out, long long total, int C,
                                   int HW) {
  const float s = ud_sigmoid(__ldg(fuse_coef));
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int pos = (int)(i % HW);
    const long long n = i / ((long long)C * HW);
    const float e = emb[i];
    const float r = res ? res[i] : e;
    out[i] = (1.f - s) * smask[n * HW + pos] * e + s * ff[i] + r;
  }
}

// grads: g_emb = (1-s)*smask*g (+ g when the residual IS emb, i.e. res was NULL in forward;
// otherwise the residual gradient is left to autograd on `res`), g_ff = s*g,
// g_smask[n,pos] = (1-s)*sum_c emb*g, g_coef = s(1-s)*sum (ff - smask*emb)*g.
// One CTA per (n, tile of 32 positions); deterministic reductions; g_coef partial per CTA.
__global__ void __launch_bounds__(256)
at_fuse_bwd_kernel(const float* __restrict__ emb, const float* __restrict__ smask, const float* __restrict__ ff,
                   const float* __restrict__ g, const float* __restrict__ fuse_coef, float* __restrict__ g_emb,
                   float* __restrict__ g_ff, float* __restrict__ g_smask, float* __restrict__ coef_part, int C, int HW,
                   int tiles, int res_is_emb) {
  __shared__ float red_m[8][33];
  __shared__ float red[33];
  const float s = ud_sigmoid(__ldg(fuse_coef));
  const int n = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;  // 8 channel groups x 32 positions
  const int pos = tile * 32 + lane;
  float gm = 0.f, gc = 0.f;
  if (pos < HW) {
    const float m = smask[(long long)n * HW + pos];
    for (int c = grp; c < C; c += 8) {
      const long long i = ((long long)n * C + c) * HW + pos;
      const float e = emb[i], gv = g[i], f = ff[i];
      g_emb[i] = (1.f - s) * m * gv + (res_is_emb ? gv : 0.f);
      g_ff[i] = s * gv;
      gm = fmaf(e, gv, gm);
      gc = fmaf(f - m * e, gv, gc);
    }
  }
  red_m[grp][lane] = gm;
  __syncthreads();
  if (grp == 0 && pos < HW) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += red_m[q][lane];
    g_smask[(long long)n * HW + pos] = (1.f - s) * t;
  }
  const float tot = ud_block_sum(gc, red);
  if (threadIdx.x == 0) coef_part[blockIdx.x] = tot * s * (1.f - s);
}

__global__ void at_sum_partials_kernel(const float* __restrict__ part, float* __restrict__ out, int n) {
  __shared__ float red[33];
  float a = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a += part[i];
  a = ud_block_sum(a, red);
  if (threadIdx.x == 0) *out = a;
}

extern "C" int ud_attn_fuse_fwd(const float* emb, const float* smask, const float* ff, const float* res,
                                const float* fuse_coef, float* out, int N, int C, int HW, cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && C >= 1 && HW >= 1, UD_ERR_INVALID, "attn_fuse_fwd: bad shape");
  const long long total = (long long)N * C * HW;
  if (total == 0) return UD_OK;
  UD_REQUIRE(emb && smask && ff && fuse_coef && out, UD_ERR_INVALID, "attn_fuse_fwd: null pointer");
  const int blocks = (int)min((long long)UD_NUM_SMS * 8, (total + 255) / 256);
  at_fuse_fwd_kernel<<<blocks, 256, 0, stream>>>(emb, smask, ff, res, fuse_coef, out, total, C, HW);
  return ud_check_launch("attn_fuse_fwd");
}

extern "C" size_t ud_attn_fuse_bwd_workspace_bytes(int N, int HW) { return sizeof(float) * (size_t)N * ud_cdiv(HW, 32); }

extern "C" int ud_attn_fuse_bwd(const float* emb, const float* smask, const float* ff, const float* g,
                                const float* fuse_coef, float* g_emb, float* g_ff, float* g_smask, float* g_coef,
                                void* ws, size_t ws_bytes, int N, int C, int HW, int res_is_emb,
                                cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && C >= 1 && HW >= 1, UD_ERR_INVALID, "attn_fuse_bwd: bad shape");
  UD_REQUIRE(g_coef, UD_ERR_INVALID, "attn_fuse_bwd: null pointer");
  if (N == 0) {
    UD_CUDA(cudaMemsetAsync(g_coef, 0, sizeof(float), stream));
    return UD_OK;
  }
  UD_REQUIRE(emb && smask && ff && g && fuse_coef && g_emb && g_ff && g_smask && ws, UD_ERR_INVALID,
             "attn_fuse_bwd: null pointer");
  UD_REQUIRE(ws_bytes >= ud_attn_fuse_bwd_workspace_bytes(N, HW), UD_ERR_WORKSPACE, "attn_fuse_bwd: workspace too small");
  const int tiles = ud_cdiv(HW, 32);
  float* part = static_cast<float*>(ws);
  at_fuse_bwd_kernel<<<N * tiles, 256, 0, stream>>>(emb, smask, ff, g, fuse_coef, g_emb, g_ff, g_smask, part, C, HW,
                                                    tiles, res_is_emb);
  int rc = ud_check_launch("attn_fuse_bwd");
  if (rc != UD_OK) return rc;
  at_sum_partials_kernel<<<1, 256, 0, stream>>>(part, g_coef, N * tiles);
  return ud_check_launch("attn_fuse_bwd_sum");
}
