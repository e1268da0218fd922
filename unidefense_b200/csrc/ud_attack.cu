// a19 -- projected-gradient attack step (PGD / FGSM robustness evaluation)
//
// One PGD iteration's image-sized work for a batch: best-iterate selection, the signed (L-inf) or normalised (L2) step,
// the projection onto the eps-ball around x0 and the clamp to the input range.  The formulas mirror the torch
// composition of oracle/attack.py operation for operation, each rounding explicit (__fadd_rn and friends), so the L-inf
// step is bit-identical to it.  Per-sample L2 norms are fixed-order: every CTA of a sample writes one partial sum into
// the workspace and the consumers add the partials in index order, so repeated calls are bitwise identical.
//
// Launches: L-inf or select-only = select prologue + elementwise pass; L2 = g-norm pass (which also selects) +
// d-norm pass + elementwise pass.  The elementwise pass reads the per-sample "improved" flag the earlier launch left in
// the workspace, never best_loss, which that launch has already updated.
#include <math.h>

#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

#define PG_THREADS 256
#define PG_CHUNK 4096   // elements of one sample per CTA: 4 float4 per thread; fixes the order of the L2 partial sums

struct PgArgs {
  const float* x0;
  float* xa;
  const float* g;
  const float* loss;
  float* best_loss;
  float* xb;
  const float* eps;
  const float* alpha;
  int* flag;     // ws: [N] improved flags
  float* gpart;  // ws: [N, chunks] partial sums of g^2
  float* dpart;  // ws: [N, chunks] partial sums of d^2
  float lo, hi;
  long long P;   // elements per sample
  int chunks;
};

// The elements CTA `c` of sample `n` owns, as float4 groups (VEC) or single elements.  With VEC the sample's first
// elements up to a 16-byte boundary (head) go to chunk 0 and the remainder after the last whole float4 (tail) to the
// last chunk; every pointer shares the same alignment, which the host checks.
struct PgRange {
  long long base;      // offset of the sample's first element
  long long head;      // scalar elements before the first float4
  long long v0, v1;    // float4 groups [v0, v1) of this chunk, counted from base + head
  long long tail0;     // first tail element (relative to base)
  bool first, last;
};

template <bool VEC>
__device__ __forceinline__ PgRange pg_range(const PgArgs& a, int n, int c) {
  PgRange r;
  r.base = (long long)n * a.P;
  r.first = c == 0;
  r.last = c == a.chunks - 1;
  if (VEC) {
    r.head = min((long long)((4 - (r.base & 3)) & 3), a.P);
    const long long nv = (a.P - r.head) >> 2;
    const long long per = PG_CHUNK / 4;
    r.v0 = min((long long)c * per, nv);
    r.v1 = min(r.v0 + per, nv);
    r.tail0 = r.head + 4 * nv;
  } else {
    r.head = 0;
    r.v0 = min((long long)c * PG_CHUNK, a.P);
    r.v1 = min(r.v0 + PG_CHUNK, a.P);
    r.tail0 = a.P;
  }
  return r;
}

// Fixed-order sum of a sample's partials, broadcast to the CTA.
__device__ __forceinline__ float pg_sum_partials(const float* part, int chunks, float* sh) {
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < chunks; ++i) s = __fadd_rn(s, part[i]);
    *sh = s;
  }
  __syncthreads();
  return *sh;
}

__device__ __forceinline__ bool pg_select(const PgArgs& a, int n) {
  const float l = a.loss[n], b = a.best_loss[n];
  const bool imp = l > b;   // strict; a NaN loss never improves
  if (imp) a.best_loss[n] = l;
  a.flag[n] = imp ? 1 : 0;
  return imp;
}

// u = g / (||g|| + 1e-12);  d = (x_adv + alpha*u) - x0
__device__ __forceinline__ float pg_l2_d(float x0, float xa, float g, float gden, float alpha) {
  return __fsub_rn(__fadd_rn(xa, __fmul_rn(alpha, __fdiv_rn(g, gden))), x0);
}

__device__ __forceinline__ float pg_clamp(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

__global__ void __launch_bounds__(PG_THREADS) pg_select_kernel(PgArgs a, int N) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) pg_select(a, n);
}

// L2 pass 1: partial sums of g^2 (and the select, by the first CTA of the sample).
template <bool VEC>
__global__ void __launch_bounds__(PG_THREADS) pg_gnorm_kernel(PgArgs a) {
  __shared__ float red[33];
  const int c = blockIdx.x, n = blockIdx.y;
  if (c == 0 && threadIdx.x == 0) pg_select(a, n);
  const PgRange r = pg_range<VEC>(a, n, c);
  const float* g = a.g + r.base;
  float s = 0.f;
  if (VEC) {
    const float4* g4 = reinterpret_cast<const float4*>(g + r.head);
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) {
      const float4 v = __ldg(g4 + i);
      s = __fmaf_rn(v.x, v.x, s);
      s = __fmaf_rn(v.y, v.y, s);
      s = __fmaf_rn(v.z, v.z, s);
      s = __fmaf_rn(v.w, v.w, s);
    }
    if (r.first && threadIdx.x < r.head) s = __fmaf_rn(g[threadIdx.x], g[threadIdx.x], s);
    if (r.last && r.tail0 + threadIdx.x < a.P) s = __fmaf_rn(g[r.tail0 + threadIdx.x], g[r.tail0 + threadIdx.x], s);
  } else {
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) s = __fmaf_rn(__ldg(g + i), __ldg(g + i), s);
  }
  s = ud_block_sum(s, red);
  if (threadIdx.x == 0) a.gpart[(long long)n * a.chunks + c] = s;
}

// L2 pass 2: partial sums of d^2, d = x_adv + alpha*g/(||g||+1e-12) - x0.
template <bool VEC>
__global__ void __launch_bounds__(PG_THREADS) pg_dnorm_kernel(PgArgs a) {
  __shared__ float red[33];
  const int c = blockIdx.x, n = blockIdx.y;
  const float gden = __fadd_rn(__fsqrt_rn(pg_sum_partials(a.gpart + (long long)n * a.chunks, a.chunks, red)), 1e-12f);
  const float al = a.alpha[n];
  const PgRange r = pg_range<VEC>(a, n, c);
  const float *x0 = a.x0 + r.base, *xa = a.xa + r.base, *g = a.g + r.base;
  float s = 0.f;
  auto one = [&](long long i) {
    const float d = pg_l2_d(__ldg(x0 + i), xa[i], __ldg(g + i), gden, al);
    s = __fmaf_rn(d, d, s);
  };
  if (VEC) {
    const float4* x04 = reinterpret_cast<const float4*>(x0 + r.head);
    const float4* xa4 = reinterpret_cast<const float4*>(xa + r.head);
    const float4* g4 = reinterpret_cast<const float4*>(g + r.head);
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) {
      const float4 p = __ldg(x04 + i), q = xa4[i], v = __ldg(g4 + i);
      float d;
      d = pg_l2_d(p.x, q.x, v.x, gden, al); s = __fmaf_rn(d, d, s);
      d = pg_l2_d(p.y, q.y, v.y, gden, al); s = __fmaf_rn(d, d, s);
      d = pg_l2_d(p.z, q.z, v.z, gden, al); s = __fmaf_rn(d, d, s);
      d = pg_l2_d(p.w, q.w, v.w, gden, al); s = __fmaf_rn(d, d, s);
    }
    if (r.first && threadIdx.x < r.head) one(threadIdx.x);
    if (r.last && r.tail0 + threadIdx.x < a.P) one(r.tail0 + threadIdx.x);
  } else {
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) one(i);
  }
  s = ud_block_sum(s, red);
  if (threadIdx.x == 0) a.dpart[(long long)n * a.chunks + c] = s;
}

// Elementwise pass: x_best = x_adv (pre-step) where the sample improved; then the step (STEP) under NORM.
template <bool VEC, bool STEP, int NORM>
__global__ void __launch_bounds__(PG_THREADS) pg_apply_kernel(PgArgs a) {
  __shared__ float red[2];
  const int c = blockIdx.x, n = blockIdx.y;
  const bool imp = a.flag[n] != 0;
  if (!STEP && !imp) return;
  float gden = 0.f, f = 1.f;
  const float al = STEP ? a.alpha[n] : 0.f, ep = STEP ? a.eps[n] : 0.f;
  if (STEP && NORM == UD_NORM_L2) {
    gden = __fadd_rn(__fsqrt_rn(pg_sum_partials(a.gpart + (long long)n * a.chunks, a.chunks, red)), 1e-12f);
    const float dn = __fsqrt_rn(pg_sum_partials(a.dpart + (long long)n * a.chunks, a.chunks, red + 1));
    f = dn > ep ? __fdiv_rn(ep, dn) : 1.f;     // min(1, eps/||d||), 0/0 -> 1
  }
  const PgRange r = pg_range<VEC>(a, n, c);
  const float* x0 = a.x0 + r.base;
  float* xa = a.xa + r.base;
  float* xb = a.xb + r.base;
  const float* g = STEP ? a.g + r.base : nullptr;
  const float lo = a.lo, hi = a.hi;
  auto step = [&](float p, float q, float v) -> float {
    float d;
    if (NORM == UD_NORM_LINF) {
      d = __fsub_rn(__fadd_rn(q, __fmul_rn(al, ud_sign(v))), p);
      d = fminf(fmaxf(d, -ep), ep);
    } else {
      d = __fmul_rn(pg_l2_d(p, q, v, gden, al), f);
    }
    return pg_clamp(__fadd_rn(p, d), lo, hi);
  };
  auto one = [&](long long i) {
    const float q = xa[i];
    if (imp) xb[i] = q;
    if (STEP) xa[i] = step(__ldg(x0 + i), q, __ldg(g + i));
  };
  if (VEC) {
    const float4* x04 = reinterpret_cast<const float4*>(x0 + r.head);
    float4* xa4 = reinterpret_cast<float4*>(xa + r.head);
    float4* xb4 = reinterpret_cast<float4*>(xb + r.head);
    const float4* g4 = reinterpret_cast<const float4*>(g + r.head);
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) {
      const float4 q = xa4[i];
      if (imp) xb4[i] = q;
      if (STEP) {
        const float4 p = __ldg(x04 + i), v = __ldg(g4 + i);
        xa4[i] = make_float4(step(p.x, q.x, v.x), step(p.y, q.y, v.y), step(p.z, q.z, v.z), step(p.w, q.w, v.w));
      }
    }
    if (r.first && threadIdx.x < r.head) one(threadIdx.x);
    if (r.last && r.tail0 + threadIdx.x < a.P) one(r.tail0 + threadIdx.x);
  } else {
#pragma unroll 4
    for (long long i = r.v0 + threadIdx.x; i < r.v1; i += PG_THREADS) one(i);
  }
}

static int pg_chunks(long long P) { return ud_cdiv(P, PG_CHUNK); }

extern "C" size_t ud_attack_workspace_bytes(int N, long long per_sample) {
  if (N < 1 || per_sample < 1) return 0;
  const size_t part = sizeof(float) * (size_t)N * (size_t)pg_chunks(per_sample);
  return ud_align_up(sizeof(int) * (size_t)N, 256) + 2 * ud_align_up(part, 256);
}

template <bool VEC>
static void pg_launch(const PgArgs& a, int norm, bool step, int N, cudaStream_t stream) {
  const dim3 grid(a.chunks, N);
  if (!step) {
    pg_apply_kernel<VEC, false, UD_NORM_LINF><<<grid, PG_THREADS, 0, stream>>>(a);
  } else if (norm == UD_NORM_LINF) {
    pg_apply_kernel<VEC, true, UD_NORM_LINF><<<grid, PG_THREADS, 0, stream>>>(a);
  } else {
    pg_apply_kernel<VEC, true, UD_NORM_L2><<<grid, PG_THREADS, 0, stream>>>(a);
  }
}

extern "C" int ud_attack_step(const float* x0, float* x_adv, const float* g, const float* loss, float* best_loss,
                              float* x_best, const float* eps, const float* alpha, float lo, float hi, int norm, int N,
                              long long per_sample, void* ws, size_t ws_bytes, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && per_sample >= 1, UD_ERR_INVALID, "attack_step: bad shape N=%d per_sample=%lld", N, per_sample);
  UD_REQUIRE(norm == UD_NORM_LINF || norm == UD_NORM_L2, UD_ERR_INVALID,
             "attack_step: unknown norm %d (UD_NORM_LINF=0, UD_NORM_L2=2)", norm);
  UD_REQUIRE(lo <= hi, UD_ERR_INVALID, "attack_step: lo=%g > hi=%g", (double)lo, (double)hi);
  UD_REQUIRE(N <= 65535, UD_ERR_UNSUPPORTED, "attack_step: N=%d > 65535", N);
  const size_t need = ud_attack_workspace_bytes(N, per_sample);
  UD_REQUIRE(ws && ws_bytes >= need, UD_ERR_WORKSPACE, "attack_step: workspace of %zu bytes, %zu needed", ws_bytes, need);
  UD_REQUIRE(x0 && x_adv && loss && best_loss && x_best, UD_ERR_INVALID, "attack_step: null pointer");
  UD_REQUIRE(!g || (eps && alpha), UD_ERR_INVALID, "attack_step: a step needs eps and alpha");

  PgArgs a;
  a.x0 = x0; a.xa = x_adv; a.g = g; a.loss = loss; a.best_loss = best_loss; a.xb = x_best; a.eps = eps; a.alpha = alpha;
  char* w = (char*)ws;
  a.flag = (int*)w;
  w += ud_align_up(sizeof(int) * (size_t)N, 256);
  a.gpart = (float*)w;
  a.dpart = (float*)(w + ud_align_up(sizeof(float) * (size_t)N * (size_t)pg_chunks(per_sample), 256));
  a.lo = lo; a.hi = hi; a.P = per_sample; a.chunks = pg_chunks(per_sample);

  // float4 groups need every tensor at the same offset from a 16-byte boundary: true for torch allocations
  const uintptr_t al = (uintptr_t)x0 | (uintptr_t)x_adv | (uintptr_t)x_best | (uintptr_t)(g ? g : x0);
  const bool vec = (al & 15) == 0;
  const bool step = g != nullptr;
  const dim3 grid(a.chunks, N);
  if (step && norm == UD_NORM_L2) {
    if (vec) {
      pg_gnorm_kernel<true><<<grid, PG_THREADS, 0, stream>>>(a);
    } else {
      pg_gnorm_kernel<false><<<grid, PG_THREADS, 0, stream>>>(a);
    }
    int rc = ud_check_launch("attack_step (g norm)");
    if (rc) return rc;
    if (vec) {
      pg_dnorm_kernel<true><<<grid, PG_THREADS, 0, stream>>>(a);
    } else {
      pg_dnorm_kernel<false><<<grid, PG_THREADS, 0, stream>>>(a);
    }
    rc = ud_check_launch("attack_step (d norm)");
    if (rc) return rc;
  } else {
    pg_select_kernel<<<ud_cdiv(N, PG_THREADS), PG_THREADS, 0, stream>>>(a, N);
    const int rc = ud_check_launch("attack_step (select)");
    if (rc) return rc;
  }
  if (vec) {
    pg_launch<true>(a, norm, step, N, stream);
  } else {
    pg_launch<false>(a, norm, step, N, stream);
  }
  return ud_check_launch("attack_step");
}
