// a22 -- Fourier-basis perturbations (Fourier heat maps of a detector's sensitivity, after Yin et al., NeurIPS 2019)
//
// ud_fourier_perturb writes y = clamp(x + r_{n,c} * eps * a * cos(2 pi k(h, w) / (H*W)), lo, hi) for the canonical
// frequency freqs[*f], in one elementwise pass (one read of x, one write of y).  f, eps and the seed are read from
// device memory, so one captured CUDA graph serves every frequency, eps and seed.  A thread owns four consecutive
// pixels of a plane: it computes their cosines once and applies them to every (sample, channel) plane of its CTA, so the
// trigonometry costs H*W*ceil(N*C/FR_PLANES) cospif rather than one per element.  Every rounding is explicit (no FMA
// contraction) and every output element is written once: bitwise reproducible.
#include <math.h>
#include <stdint.h>

#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"
#include "ud_philox.cuh"

#define FR_THREADS 256
#define FR_PLANES 16              // (sample, channel) planes per CTA
#define FR_SIGN_TAG 0x464F5552u   // "FOUR"; distinct from ud_corrupt's and ud_explain's tags

// VEC: every plane of x and y starts on a 16-byte boundary (both pointers aligned and H*W % 4 == 0), so each thread's
// four pixels are one float4 in every plane.  Otherwise a plane takes the float4 path only where both of its starts
// are aligned, and scalar loads elsewhere.  The last group of a plane (H*W % 4 pixels) is scalar either way.
template <bool VEC>
__global__ void __launch_bounds__(FR_THREADS)
    fr_perturb_kernel(const float* __restrict__ x, float* __restrict__ y, const int* __restrict__ freqs, int F,
                      const int* fp, const float* epsp, const long long* __restrict__ ids,
                      const unsigned long long* seedp, float lo, float hi, float a_half, float a_full, int C, int H,
                      int W, long long HW, int planes) {
  __shared__ float s_sh[FR_PLANES];
  const int fi = *fp;
  if (fi < 0 || fi >= F) return;
  const int uu = __ldg(freqs + 2 * fi), vv = __ldg(freqs + 2 * fi + 1);
  if (uu < 0 || uu >= H || vv < 0 || vv >= W) return;
  const int p0 = blockIdx.x * FR_PLANES;
  const int np = min(FR_PLANES, planes - p0);
  if (threadIdx.x < np) {
    // s = r * (eps * a): the sign r_{n,c} is bit (c & 31) of word (c >> 5) of the sample's Philox block
    const int p = p0 + threadIdx.x, n = p / C, c = p - n * C;
    const unsigned long long id = ids ? (unsigned long long)ids[n] : (unsigned long long)n;
    const unsigned long long sd = *seedp;
    const uint4 r = ud_philox(make_uint4(((unsigned)uu << 16) | (unsigned)vv, (unsigned)id, (unsigned)(id >> 32), 0u),
                              (unsigned)sd, (unsigned)(sd >> 32) ^ FR_SIGN_TAG);
    const int wd = c >> 5;
    const unsigned word = wd == 0 ? r.x : wd == 1 ? r.y : wd == 2 ? r.z : r.w;
    const bool self_conj = (2 * uu) % H == 0 && (2 * vv) % W == 0;        // DC and the Nyquist corners
    const float m = __fmul_rn(*epsp, self_conj ? a_half : a_full);
    s_sh[threadIdx.x] = ((word >> (c & 31)) & 1u) ? -m : m;
  }
  __syncthreads();
  const long long q0 = 4LL * ((long long)blockIdx.y * FR_THREADS + threadIdx.x);
  if (q0 >= HW) return;
  const int nq = (int)min(4LL, HW - q0);
  float cs[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    cs[i] = 0.f;
    if (i < nq) {
      const int q = (int)q0 + i, h = q / W, w = q - h * W;
      const int k = (int)(((long long)((uu * h) % H) * W + (long long)((vv * w) % W) * H) % HW);
      const float t = __fdiv_rn((float)k, (float)HW);                       // turns; k and H*W <= 2^24 are exact
      cs[i] = cospif(__fmul_rn(2.f, t));
    }
  }
  auto one = [&](float xv, float s, float cv) { return fminf(fmaxf(__fadd_rn(xv, __fmul_rn(s, cv)), lo), hi); };
  if (VEC && nq == 4) {
    const float4* x4 = reinterpret_cast<const float4*>(x + (long long)p0 * HW + q0);
    float4* y4 = reinterpret_cast<float4*>(y + (long long)p0 * HW + q0);
    const long long st = HW >> 2;
#pragma unroll 4
    for (int j = 0; j < np; ++j) {
      const float s = s_sh[j];
      const float4 v = __ldg(x4 + j * st);
      y4[j * st] = make_float4(one(v.x, s, cs[0]), one(v.y, s, cs[1]), one(v.z, s, cs[2]), one(v.w, s, cs[3]));
    }
    return;
  }
  for (int j = 0; j < np; ++j) {
    const float s = s_sh[j];
    const long long o = (long long)(p0 + j) * HW + q0;
    if (nq == 4 && (((uintptr_t)(x + o) | (uintptr_t)(y + o)) & 15) == 0) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + o));
      *reinterpret_cast<float4*>(y + o) =
          make_float4(one(v.x, s, cs[0]), one(v.y, s, cs[1]), one(v.z, s, cs[2]), one(v.w, s, cs[3]));
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < nq) y[o + i] = one(__ldg(x + o + i), s, cs[i]);
    }
  }
}

extern "C" int ud_fourier_perturb(const float* x, float* y, const int* freqs, int F, const int* f, const float* eps,
                                  const long long* ids, const unsigned long long* seed, float lo, float hi, int N, int C,
                                  int H, int W, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && C >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "fourier_perturb: bad shape N=%d C=%d H=%d W=%d",
             N, C, H, W);
  UD_REQUIRE(N <= 65535, UD_ERR_UNSUPPORTED, "fourier_perturb: N=%d > 65535", N);
  UD_REQUIRE(C <= 128, UD_ERR_UNSUPPORTED, "fourier_perturb: C=%d > 128 (one sign bit per channel of a Philox block)",
             C);
  const long long HW = (long long)H * W;
  UD_REQUIRE(H <= 4096 && W <= 4096 && HW <= (1LL << 24), UD_ERR_UNSUPPORTED,
             "fourier_perturb: H=%d, W=%d: needs H, W <= 4096 and H*W <= 2^24 (an exact fp32 phase)", H, W);
  UD_REQUIRE(F >= 1, UD_ERR_INVALID, "fourier_perturb: F=%d < 1 (the frequency table's length)", F);
  UD_REQUIRE(x && y && freqs && f && eps && seed, UD_ERR_INVALID, "fourier_perturb: null pointer");
  UD_REQUIRE(lo <= hi, UD_ERR_INVALID, "fourier_perturb: need lo <= hi, got lo=%g hi=%g", (double)lo, (double)hi);
  const long long planes = (long long)N * C;
  const uintptr_t bytes = (uintptr_t)(planes * HW) * sizeof(float);
  UD_REQUIRE((uintptr_t)y + bytes <= (uintptr_t)x || (uintptr_t)x + bytes <= (uintptr_t)y, UD_ERR_INVALID,
             "fourier_perturb: y overlaps x");

  const float a_half = (float)sqrt(1.0 / (double)HW), a_full = (float)sqrt(2.0 / (double)HW);
  const dim3 grid(ud_cdiv(planes, FR_PLANES), ud_cdiv(HW, 4LL * FR_THREADS));
  const bool vec = ((((uintptr_t)x | (uintptr_t)y) & 15) == 0) && (HW & 3) == 0;
  if (vec) {
    fr_perturb_kernel<true><<<grid, FR_THREADS, 0, stream>>>(x, y, freqs, F, f, eps, ids, seed, lo, hi, a_half, a_full,
                                                             C, H, W, HW, (int)planes);
  } else {
    fr_perturb_kernel<false><<<grid, FR_THREADS, 0, stream>>>(x, y, freqs, F, f, eps, ids, seed, lo, hi, a_half,
                                                              a_full, C, H, W, HW, (int)planes);
  }
  return ud_check_launch("fourier_perturb");
}
