// Line FFT of ANY length 1 <= n <= UD_FFT_MAX_N for the shared-memory kernels (sm_100a).
//
// n whose prime factors are all <= 23 runs the mixed-radix Stockham stages of ud_fft.cuh (UdDynPlan).  Every other
// n (29, 31, 37 ... as a factor: 58, 62, 248, 372 ...) runs Bluestein's chirp-z algorithm on top of the same
// stages: with w[j] = exp(-i pi j^2 / n),
//     X[k] = w[k] * sum_j (x[j] w[j]) * conj(w)[k - j]
// is a linear convolution, evaluated as a circular one of power-of-two length m >= 2n-1:
//     A = FFT_m(x.w zero-padded),  C = A * Bhat,  c = IFFT_m(C) = conj(FFT_m(conj C)) / m,  X[k] = w[k] c[k]
// where Bhat = FFT_m(conj(w) wrapped to length m) / m is a per-(device, n) table computed on the host in double
// precision (the phase j^2 mod 2n is reduced in integer arithmetic, so the chirp is accurate to fp32 rounding).
// The north star asks for "mixed-radix/Bluestein for non-power-of-two sizes"; the reference itself accepts any size
// because torch.fft does (model/unidefense.py:246-249, model/modules.py:43-54).
//
// A line buffer holds line_len() = m complex points (m = n for mixed radix); the plan always ping-pongs between two
// buffers.  Forward sign only; callers obtain the inverse with the re/im swap trick.
#pragma once
#include "ud_fft.cuh"

struct UdAnyPlan {
  static constexpr bool kInPlace = false;
  int n_;                // logical line length
  int m;                 // working length: n, or Bluestein's power of two >= 2n-1
  int bluestein;
  UdDynPlan inner;       // Stockham stages of length m
  const float2* tw;      // device: exp(-2 pi i t / m), t < m
  const float2* chirp;   // device (Bluestein): w[j], j < n
  const float2* bhat;    // device (Bluestein): FFT_m(wrapped conj chirp) / m

  __device__ __forceinline__ int n() const { return n_; }
  __device__ __forceinline__ int line_len() const { return m; }

  // Forward DFT of L lines held in `a` (n valid points per line, line stride LS >= m); `tw_s` = the m twiddles staged
  // in shared memory.  Data must be visible (caller synced).  Returns the buffer holding the n results per line;
  // ends with a __syncthreads().
  __device__ __forceinline__ float2* run(float2* a, float2* b, const float2* tw_s, int L, int LS) const {
    if (!bluestein) return inner.run(a, b, tw_s, L, LS);
    const int n = n_;
    for (int idx = threadIdx.x; idx < L * m; idx += blockDim.x) {
      const int line = idx / m, j = idx - line * m;
      float2* p = a + line * LS + j;
      *p = (j < n) ? ud_cmul(*p, __ldg(chirp + j)) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    float2* r = inner.run(a, b, tw_s, L, LS);
    float2* o = (r == a) ? b : a;
    for (int idx = threadIdx.x; idx < L * m; idx += blockDim.x) {
      const int line = idx / m, k = idx - line * m;
      float2* p = r + line * LS + k;
      const float2 c = ud_cmul(*p, __ldg(bhat + k));
      *p = make_float2(c.x, -c.y);
    }
    __syncthreads();
    float2* r2 = inner.run(r, o, tw_s, L, LS);
    for (int idx = threadIdx.x; idx < L * n; idx += blockDim.x) {
      const int line = idx / n, k = idx - line * n;
      float2* p = r2 + line * LS + k;
      *p = ud_cmul(make_float2(p->x, -p->y), __ldg(chirp + k));
    }
    __syncthreads();
    return r2;
  }
};

// Host: fills `plan` for any 1 <= n <= UD_FFT_MAX_N (tables cached per (device, n), created on first use -- not
// during a CUDA-graph capture).  Returns false (error set) on failure.
bool ud_make_any_plan(int n, UdAnyPlan* plan);
// Host: the working length m of n's plan (n, or Bluestein's power of two >= 2n-1) without creating the plan; 0 outside
// [1, UD_FFT_MAX_N].
int ud_any_line_len(int n);
// odd line stride for a plan's line buffers
static inline int ud_any_line_stride(const UdAnyPlan& p) { return p.m | 1; }

// Host: lines per CTA of a kernel that keeps two ping-pong buffers of (m | 1) points per line: the largest L <= lmax for
// which `fixed` bytes (staged twiddles, tables) plus L * (two line buffers + `per_line` other bytes) fit in `budget`
// bytes; 0 when not even one line fits.  Every shared-memory line-FFT kernel sizes its lines here.
static inline int ud_any_lines(int m, size_t fixed, size_t per_line, size_t budget, int lmax) {
  const size_t line = 2 * sizeof(float2) * (size_t)(m | 1) + per_line;
  if (budget < fixed + line) return 0;
  const size_t L = (budget - fixed) / line;
  return L < (size_t)lmax ? (int)L : lmax;
}
// Kernels instantiated at lmax, lmax/2 and lmax/4 lines per CTA: the largest of those <= fit (a ud_any_lines result);
// 0 when none is.
static inline int ud_halving_lines(int fit, int lmax) {
  for (int L = lmax; L >= lmax / 4 && L >= 1; L /= 2)
    if (L <= fit) return L;
  return 0;
}
// runs the body with `constexpr int LV` bound to L, which is one of X, X/2 and X/4 (a ud_halving_lines result)
#define UD_LINES_DISPATCH(L, X, LV, ...)                                 \
  do {                                                                   \
    if ((L) == (X)) { constexpr int LV = (X); __VA_ARGS__; }             \
    else if ((L) == (X) / 2) { constexpr int LV = (X) / 2; __VA_ARGS__; } \
    else { constexpr int LV = (X) / 4; __VA_ARGS__; }                    \
  } while (0)
