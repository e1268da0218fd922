// Shared-memory line FFT building blocks (mixed radix Stockham autosort) for sm_100a.
//
// A "line" is one complex sequence of length n held in shared memory as float2.  A CTA keeps
// L lines resident (line stride LS float2, LS odd so transposing loads are bank-conflict
// free) and runs every stage over all of them; one thread owns one radix-R butterfly at a
// time.  n = R0*R1*...; stage s (radix R, Ns = product of earlier radices):
//     v[r]  = in[j + r*n/R] * W_n^(r * (j mod Ns) * n/(Ns*R))       r = 0..R-1
//     v     = DFT_R(v)
//     out[(j div Ns)*Ns*R + (j mod Ns) + r*Ns] = v[r]
// Natural order in, natural order out, ping-pong between two buffers.  Forward sign only;
// the inverse is obtained by the callers by swapping re/im on load and store.
//
// Plans: UdStaticPlanIP<N, L, THREADS, R0, R1, ...> (in place, all index arithmetic constant-folded) for the
// configured lengths (UdConfigured below) and UdDynPlan for any n whose prime factors are <= 23.  The configured
// lengths also have a register-resident two-stage plan (Ud2S).
#pragma once
#include "ud_common.cuh"
#include "ud_fft_bfly_gen.cuh"

#define UD_FFT_MAX_STAGES 10

__device__ __forceinline__ float2 ud_cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// Radix-R butterfly, forward sign, in place: the generated straight-line code of ud_fft_bfly_gen.cuh
template <int R>
struct UdBfly;
#define UD_BFLY(R)                                                                \
  template <>                                                                     \
  struct UdBfly<R> {                                                              \
    static __device__ __forceinline__ void run(float2 (&v)[R]) { ud_bfly##R(v); } \
  };
UD_BFLY(2) UD_BFLY(3) UD_BFLY(4) UD_BFLY(5) UD_BFLY(7) UD_BFLY(8) UD_BFLY(11) UD_BFLY(12) UD_BFLY(13) UD_BFLY(14)
UD_BFLY(16) UD_BFLY(17) UD_BFLY(19) UD_BFLY(20) UD_BFLY(23)
#undef UD_BFLY

// One Stockham stage over L lines.  tw[t] = exp(-2 pi i t / n), t in [0, n).
template <int R>
__device__ __forceinline__ void ud_fft_stage(const float2* __restrict__ in, float2* __restrict__ out,
                                             const float2* __restrict__ tw, const int n, const int Ns,
                                             const int L, const int LS) {
  const int T = n / R;          // butterflies per line
  const int tstride = T / Ns;   // n / (Ns*R)
  const int total = L * T;
  for (int wi = threadIdx.x; wi < total; wi += blockDim.x) {
    const int line = wi / T;
    const int j = wi - line * T;
    const int q = j / Ns;
    const int k = j - q * Ns;
    const float2* src = in + line * LS + j;
    float2 v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = src[r * T];
    if (Ns > 1) {
      const int t1 = k * tstride;
#pragma unroll
      for (int r = 1; r < R; ++r) v[r] = ud_cmul(v[r], tw[r * t1]);
    }
    UdBfly<R>::run(v);
    float2* dst = out + line * LS + q * Ns * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) dst[r * Ns] = v[r];
  }
}

// ---- plans ---------------------------------------------------------------------------
struct UdDynPlan {
  static constexpr bool kInPlace = false;
  int n_;
  int nstages;
  int radix[UD_FFT_MAX_STAGES];
  __device__ __forceinline__ int n() const { return n_; }
  __device__ __forceinline__ int line_len() const { return n_; }
  __device__ __forceinline__ float2* run(float2* a, float2* b, const float2* tw, int L, int LS) const {
    int Ns = 1;
    for (int s = 0; s < nstages; ++s) {
      const int R = radix[s];
      switch (R) {
        case 2: ud_fft_stage<2>(a, b, tw, n_, Ns, L, LS); break;
        case 3: ud_fft_stage<3>(a, b, tw, n_, Ns, L, LS); break;
        case 4: ud_fft_stage<4>(a, b, tw, n_, Ns, L, LS); break;
        case 5: ud_fft_stage<5>(a, b, tw, n_, Ns, L, LS); break;
        case 7: ud_fft_stage<7>(a, b, tw, n_, Ns, L, LS); break;
        case 11: ud_fft_stage<11>(a, b, tw, n_, Ns, L, LS); break;
        case 13: ud_fft_stage<13>(a, b, tw, n_, Ns, L, LS); break;
        case 17: ud_fft_stage<17>(a, b, tw, n_, Ns, L, LS); break;
        case 19: ud_fft_stage<19>(a, b, tw, n_, Ns, L, LS); break;
        default: ud_fft_stage<23>(a, b, tw, n_, Ns, L, LS); break;
      }
      __syncthreads();
      Ns *= R;
      float2* t = a;
      a = b;
      b = t;
    }
    return a;
  }
};

// ---- in-place static plans ------------------------------------------------------------------
// Same Stockham stages, but ONE buffer: every thread first pulls all of its butterflies for the stage
// into registers, the CTA synchronises, then results are written back in autosort order.  Halves the
// shared memory per CTA (=> twice the resident CTAs per SM) at the price of one extra barrier per
// stage.  N, L (lines per CTA) and THREADS are compile-time so every index is constant-folded.
template <int R, int N, int NS, int L, int THREADS>
__device__ __forceinline__ void ud_fft_stage_ip(float2* __restrict__ buf, const float2* __restrict__ tw) {
  constexpr int T = N / R;
  constexpr int TOTAL = L * T;
  constexpr int PASSES = (TOTAL + THREADS - 1) / THREADS;
  constexpr int LS = N | 1;
  constexpr int TS = T / NS;
  constexpr bool FULL = (PASSES * THREADS == TOTAL);
  float2 v[PASSES][R];
#pragma unroll
  for (int p = 0; p < PASSES; ++p) {
    const int wi = (int)threadIdx.x + p * THREADS;
    if (FULL || wi < TOTAL) {
      const int line = wi / T;
      const int j = wi - line * T;
      const float2* src = buf + line * LS + j;
#pragma unroll
      for (int r = 0; r < R; ++r) v[p][r] = src[r * T];
    }
  }
  __syncthreads();
#pragma unroll
  for (int p = 0; p < PASSES; ++p) {
    const int wi = (int)threadIdx.x + p * THREADS;
    if (FULL || wi < TOTAL) {
      const int line = wi / T;
      const int j = wi - line * T;
      const int q = j / NS;
      const int k = j - q * NS;
      if (NS > 1) {
        const int t1 = k * TS;
#pragma unroll
        for (int r = 1; r < R; ++r) v[p][r] = ud_cmul(v[p][r], tw[r * t1]);
      }
      UdBfly<R>::run(v[p]);
      float2* dst = buf + line * LS + q * (NS * R) + k;
#pragma unroll
      for (int r = 0; r < R; ++r) dst[r * NS] = v[p][r];
    }
  }
  __syncthreads();
}

template <int N, int NS, int L, int THREADS, int... Rs>
struct UdIpStages;
template <int N, int NS, int L, int THREADS>
struct UdIpStages<N, NS, L, THREADS> {
  static __device__ __forceinline__ void run(float2*, const float2*) {}
};
template <int N, int NS, int L, int THREADS, int R0, int... Rest>
struct UdIpStages<N, NS, L, THREADS, R0, Rest...> {
  static __device__ __forceinline__ void run(float2* buf, const float2* tw) {
    ud_fft_stage_ip<R0, N, NS, L, THREADS>(buf, tw);
    UdIpStages<N, NS * R0, L, THREADS, Rest...>::run(buf, tw);
  }
};

// Plan concept used by the kernels:  kInPlace, n(), line_len() (>= n: the points a line buffer and the staged twiddle
// table must hold -- Bluestein plans work at a longer length), run(a, b, tw, L, LS) -> buffer holding the result.
template <int N, int L, int THREADS, int... Rs>
struct UdStaticPlanIP {
  static constexpr bool kInPlace = true;
  __device__ __forceinline__ int n() const { return N; }
  __device__ __forceinline__ int line_len() const { return N; }
  __device__ __forceinline__ float2* run(float2* a, float2*, const float2* tw, int, int) const {
    UdIpStages<N, 1, L, THREADS, Rs...>::run(a, tw);
    return a;
  }
};

// ---- register-resident two-stage plans -----------------------------------------------------------
// A line of N = R1 * R2 complex points is owned by TL = max(R1, R2) threads.  Cooley-Tukey, decimation in time:
//     n = R2*n1 + n2,  k = k1 + R1*k2
//     stage A: thread n2 (< R2) holds x[n2 + R2*n1], n1 = 0..R1-1 in registers, runs ONE radix-R1 butterfly
//              (generated straight-line code with literal twiddles), multiplies by W_N^(n2*k1) and writes
//              S[k1*P + n2] to shared memory (P = R2|1: conflict-free for the column reads that follow);
//     stage B: thread k1 (< R1) reads S[k1*P + n2], n2 = 0..R2-1, runs ONE radix-R2 butterfly and holds
//              X[k1 + R1*k2], k2 = 0..R2-1.
// One shared-memory exchange and one barrier per line instead of one per radix stage, no index arithmetic inside
// the butterflies (a thread's role is fixed), and global loads/stores happen straight from/to the registers the
// butterflies use: for a fixed n1 (k2) the TL threads of a line touch R2 (R1) consecutive elements.
// Forward sign only; callers obtain the inverse with the re/im swap trick.
template <int N_, int R1_, int R2_>
struct Ud2S {
  static_assert(R1_ * R2_ == N_, "N = R1 * R2");
  static constexpr int N = N_, R1 = R1_, R2 = R2_;
  static constexpr int TL = R1_ > R2_ ? R1_ : R2_;                     // threads per line
  static constexpr int P = R2_ | 1;                                    // pitch of the exchange layout
  static constexpr int LS = ((R1_ * P > N_ ? R1_ * P : N_) | 1);       // float2 slots of one line buffer
};

// tw2[k1*P + n2] = exp(-2 pi i n2 k1 / N), from the library's global table tw_g[t] = exp(-2 pi i t / N)
template <class PL>
__device__ __forceinline__ void ud2s_build_tw(float2* __restrict__ tw2, const float2* __restrict__ tw_g) {
  for (int t = threadIdx.x; t < PL::R1 * PL::P; t += blockDim.x) {
    const int k1 = t / PL::P, n2 = t - k1 * PL::P;
    tw2[t] = (n2 < PL::R2) ? __ldg(tw_g + n2 * k1) : make_float2(0.f, 0.f);
  }
}

// stage A on the thread's R1 values (z[n1] = x[n2 + R2*n1]); results go to the line's exchange buffer S
template <class PL>
__device__ __forceinline__ void ud2s_stage_a(float2 (&z)[PL::R1], int n2, const float2* __restrict__ tw2,
                                             float2* __restrict__ S) {
  UdBfly<PL::R1>::run(z);
  S[n2] = z[0];
#pragma unroll
  for (int k1 = 1; k1 < PL::R1; ++k1) {
    const float2 t = tw2[k1 * PL::P + n2];
    S[k1 * PL::P + n2] = make_float2(z[k1].x * t.x - z[k1].y * t.y, z[k1].x * t.y + z[k1].y * t.x);
  }
}

// stage B: u[k2] = X[k1 + R1*k2]
template <class PL>
__device__ __forceinline__ void ud2s_stage_b(float2 (&u)[PL::R2], int k1, const float2* __restrict__ S) {
#pragma unroll
  for (int n2 = 0; n2 < PL::R2; ++n2) u[n2] = S[k1 * PL::P + n2];
  UdBfly<PL::R2>::run(u);
}

// ---- configured lengths -------------------------------------------------------------------------------
// The image sizes of the reference's configs (SURVEY.md App. A.1) get compile-time plans: the in-place Stockham plan
// IP<L, THREADS> (L lines per CTA) and the two-stage plan TwoStage.  Every other length runs a run-time plan.
template <int N>
struct UdConfigured;
template <>
struct UdConfigured<380> {
  template <int L, int T> using IP = UdStaticPlanIP<380, L, T, 19, 5, 4>;
  using TwoStage = Ud2S<380, 20, 19>;
};
template <>
struct UdConfigured<256> {
  template <int L, int T> using IP = UdStaticPlanIP<256, L, T, 4, 4, 4, 4>;
  using TwoStage = Ud2S<256, 16, 16>;
};
template <>
struct UdConfigured<224> {
  template <int L, int T> using IP = UdStaticPlanIP<224, L, T, 7, 4, 4, 2>;
  using TwoStage = Ud2S<224, 16, 14>;
};
template <>
struct UdConfigured<299> {
  template <int L, int T> using IP = UdStaticPlanIP<299, L, T, 23, 13>;
  using TwoStage = Ud2S<299, 13, 23>;
};
// Runs the body with the type `CFG` bound to UdConfigured<n> when n is a configured length, and `other` otherwise.
#define UD_FFT_CONFIGURED(n, CFG, other, ...)                              \
  do {                                                                     \
    if ((n) == 380) { using CFG = UdConfigured<380>; __VA_ARGS__; }        \
    else if ((n) == 256) { using CFG = UdConfigured<256>; __VA_ARGS__; }   \
    else if ((n) == 224) { using CFG = UdConfigured<224>; __VA_ARGS__; }   \
    else if ((n) == 299) { using CFG = UdConfigured<299>; __VA_ARGS__; }   \
    else { other; }                                                        \
  } while (0)
static inline bool ud_fft_configured(int n) {
  UD_FFT_CONFIGURED(n, CFG, return false, return true);
}

// ---- host side -----------------------------------------------------------------------
// Factorises n into supported radices (largest odd primes first, then 4s, then a 2).
// Returns false when n has a prime factor > 23.
bool ud_make_dyn_plan(int n, UdDynPlan* plan);
// Device twiddle table exp(-2 pi i t/n), t in [0,n), cached per (device, n) for the process
// lifetime (mutex-guarded, never freed).  nullptr on failure (error set).
const float2* ud_twiddles(int n);
// align_corners=True bilinear table for resizing `in` -> `out` samples along one axis:
// entry d = { __int_as_float(i0), l1 } with ATen's fp32 arithmetic (scale=(in-1)/(out-1), src=scale*d,
// i0=(int)src, l1=src-i0); i1 = i0 + (i0 < in-1), l0 = 1-l1.  Cached per (device, in, out) like the twiddles.
const float2* ud_lerp_table(int in, int out);
// For the transposed resize: entry j (0 <= j < in) = {first, last} output sample whose taps (i0 or i1)
// include input sample j; first > last when none does.  Derived from the same fp32 table.
const int2* ud_lerp_ranges(int in, int out);
