// a21 -- attribution maps (Integrated Gradients, SmoothGrad) and the deletion / insertion faithfulness inputs
//
// ud_attrib_step is one iteration's image-sized work for a batch, in one elementwise pass: acc (+)= w_k * g_k, then
// the next path point p_{k+1} = b + alpha_{k+1}*(x - b) (+ sigma*eps_{k+1} for SmoothGrad), or on the last step the
// attribution (x - b)*acc (IG) / acc (SmoothGrad).  k, alpha, w, sigma and the seed are read from device memory, so
// one captured CUDA graph serves every step and every parameter value.  Every rounding is explicit (__fadd_rn and
// friends, no FMA contraction), so the IG points and the accumulation are bit-identical to the fp32 torch composition
// of oracle/explain.py.  The map sum_c |attr_c| takes a second, pixel-major launch that runs only on the last step.
// ud_attrib_mask builds the deletion or insertion input of curve point j from the per-pixel rank of the map
// (ud_rank_desc, in ud_style_sort.cu).  Every output element is written once: bitwise reproducible.
#include <math.h>

#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"
#include "ud_philox.cuh"

#define EX_THREADS 256
#define EX_CHUNK 4096             // elements of one sample per CTA: 4 float4 per thread
#define EX_NOISE_TAG 0x534D5448u  // "SMTH"; distinct from ud_corrupt's tags

struct ExArgs {
  const float* x;
  const float* b;     // baseline [N, P], or NULL: bval everywhere
  const float* g;     // NULL: the start call (acc = 0, write p_k)
  float* acc;
  float* p;
  float* attr;
  float* map;
  const int* k;
  const float* alpha;
  const float* w;
  const float* sigma;
  const long long* ids;
  const unsigned long long* seed;
  float bval;
  long long P;        // elements per sample, C*H*W
  long long HW;
  int C, S, chunks;
};

// The normals of elements 4q..4q+3 of a sample at draw k
__device__ __forceinline__ float4 ex_normals(unsigned q, unsigned idl, unsigned idh, unsigned k, unsigned s0, unsigned s1) {
  const uint4 u = ud_philox(make_uint4(q, idl, idh, k), s0, s1 ^ EX_NOISE_TAG);
  const float2 z01 = ud_box_muller(u.x, u.y), z23 = ud_box_muller(u.z, u.w);
  return make_float4(z01.x, z01.y, z23.x, z23.y);
}

__device__ __forceinline__ float ex_lane(const float4& v, int i) {
  return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
}

// element j (0..7) of the concatenation (v0, v1)
__device__ __forceinline__ float ex_lane8(const float4& v0, const float4& v1, int j) {
  return j < 4 ? ex_lane(v0, j) : ex_lane(v1, j - 4);
}

// VEC: float4 groups; the sample's elements up to a 16-byte boundary (head) go to chunk 0 and those after the last
// whole float4 (tail) to the last chunk.  Every pointer is 16-byte aligned, which the host checks.
template <bool VEC, bool SG, bool TB>
__global__ void __launch_bounds__(EX_THREADS) ex_step_kernel(ExArgs a) {
  const int k = *a.k;
  if (k < 0 || k >= a.S) return;
  const bool start = a.g == nullptr;
  const bool last = !start && k == a.S - 1;
  const int kp = start ? k : k + 1;                 // the point this call writes
  const float w = start ? 0.f : __ldg(a.w + k);
  const float al = last ? 0.f : __ldg(a.alpha + kp);
  const float sg = SG && !last ? *a.sigma : 0.f;
  const int c = blockIdx.x, n = blockIdx.y;
  const long long base = (long long)n * a.P;
  unsigned idl = 0, idh = 0, s0 = 0, s1 = 0;
  if (SG) {
    const unsigned long long id = a.ids ? (unsigned long long)a.ids[n] : (unsigned long long)n;
    const unsigned long long sd = *a.seed;
    idl = (unsigned)id; idh = (unsigned)(id >> 32);
    s0 = (unsigned)sd; s1 = (unsigned)(sd >> 32);
  }
  const float* x = a.x + base;
  const float* b = TB ? a.b + base : nullptr;
  const float* g = start ? nullptr : a.g + base;
  float* acc = a.acc + base;
  float* p = a.p + base;
  float* attr = a.attr + base;
  const float bv = a.bval;

  // one element: xv, bv, gv, old acc, its noise z -> writes acc and p, or attr
  auto elem = [&](float xv, float b_, float gv, float ac, float z, float& acc_out, float& out) {
    const float s = start ? 0.f : __fadd_rn(ac, __fmul_rn(w, gv));
    acc_out = s;
    if (last) {
      out = SG ? s : __fmul_rn(__fsub_rn(xv, b_), s);
    } else {
      float q = __fadd_rn(b_, __fmul_rn(al, __fsub_rn(xv, b_)));
      if (SG) q = __fadd_rn(q, __fmul_rn(sg, z));
      out = q;
    }
  };
  auto one = [&](long long i) {
    const float z = SG && !last ? ex_lane(ex_normals((unsigned)(i >> 2), idl, idh, (unsigned)kp, s0, s1), (int)(i & 3)) : 0.f;
    float s, o;
    elem(__ldg(x + i), TB ? __ldg(b + i) : bv, start ? 0.f : __ldg(g + i), start ? 0.f : acc[i], z, s, o);
    if (!last) acc[i] = s;
    (last ? attr : p)[i] = o;
  };

  if (VEC) {
    const long long head = min((long long)((4 - (base & 3)) & 3), a.P);
    const long long nv = (a.P - head) >> 2;
    const long long v0 = min((long long)c * (EX_CHUNK / 4), nv), v1 = min(v0 + EX_CHUNK / 4, nv);
    const float4* x4 = reinterpret_cast<const float4*>(x + head);
    const float4* b4 = reinterpret_cast<const float4*>(TB ? b + head : x);
    const float4* g4 = reinterpret_cast<const float4*>(start ? x : g + head);
    float4* acc4 = reinterpret_cast<float4*>(acc + head);
    float4* out4 = reinterpret_cast<float4*>((last ? attr : p) + head);
    const int sh = (int)(head & 3);                 // element 4v + head lies at lane (4v + head) & 3 of its Philox group
#pragma unroll 2
    for (long long v = v0 + threadIdx.x; v < v1; v += EX_THREADS) {
      const float4 xv = __ldg(x4 + v);
      const float4 bq = TB ? __ldg(b4 + v) : make_float4(bv, bv, bv, bv);
      const float4 gv = start ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(g4 + v);
      const float4 av = start ? make_float4(0.f, 0.f, 0.f, 0.f) : acc4[v];
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (SG && !last) {
        const long long e0 = head + 4 * v;
        const float4 n0 = ex_normals((unsigned)(e0 >> 2), idl, idh, (unsigned)kp, s0, s1);
        if (sh == 0) {
          z = n0;
        } else {
          const float4 n1 = ex_normals((unsigned)(e0 >> 2) + 1u, idl, idh, (unsigned)kp, s0, s1);
          z = make_float4(ex_lane8(n0, n1, sh), ex_lane8(n0, n1, sh + 1), ex_lane8(n0, n1, sh + 2), ex_lane8(n0, n1, sh + 3));
        }
      }
      float4 s, o;
      elem(xv.x, bq.x, gv.x, av.x, z.x, s.x, o.x);
      elem(xv.y, bq.y, gv.y, av.y, z.y, s.y, o.y);
      elem(xv.z, bq.z, gv.z, av.z, z.z, s.z, o.z);
      elem(xv.w, bq.w, gv.w, av.w, z.w, s.w, o.w);
      if (!last) acc4[v] = s;
      out4[v] = o;
    }
    if (c == 0 && threadIdx.x < head) one(threadIdx.x);
    if (c == a.chunks - 1 && head + 4 * nv + threadIdx.x < a.P) one(head + 4 * nv + threadIdx.x);
  } else {
    const long long i0 = min((long long)c * EX_CHUNK, a.P), i1 = min(i0 + EX_CHUNK, a.P);
#pragma unroll 4
    for (long long i = i0 + threadIdx.x; i < i1; i += EX_THREADS) one(i);
  }
}

// map[n, pix] = sum_c |attr[n, c, pix]| in channel order; only on the last step
__global__ void __launch_bounds__(EX_THREADS) ex_map_kernel(ExArgs a) {
  if (*a.k != a.S - 1) return;
  const long long pix = (long long)blockIdx.x * EX_THREADS + threadIdx.x;
  if (pix >= a.HW) return;
  const int n = blockIdx.y;
  const float* at = a.attr + (long long)n * a.P + pix;
  float m = 0.f;
  for (int c = 0; c < a.C; ++c) m = __fadd_rn(m, fabsf(at[(long long)c * a.HW]));
  a.map[(long long)n * a.HW + pix] = m;
}

template <bool VEC>
static void ex_launch(const ExArgs& a, int method, int N, cudaStream_t stream) {
  const dim3 grid(a.chunks, N);
  const bool sg = method == UD_ATTRIB_SMOOTHGRAD, tb = a.b != nullptr;
  if (sg && tb) {
    ex_step_kernel<VEC, true, true><<<grid, EX_THREADS, 0, stream>>>(a);
  } else if (sg) {
    ex_step_kernel<VEC, true, false><<<grid, EX_THREADS, 0, stream>>>(a);
  } else if (tb) {
    ex_step_kernel<VEC, false, true><<<grid, EX_THREADS, 0, stream>>>(a);
  } else {
    ex_step_kernel<VEC, false, false><<<grid, EX_THREADS, 0, stream>>>(a);
  }
}

extern "C" int ud_attrib_step(const float* x, const float* base, float base_value, const float* g, float* acc, float* p,
                              float* attr, float* map, const int* k, const float* alpha, const float* w,
                              const float* sigma, const long long* ids, const unsigned long long* seed, int steps,
                              int method, int N, int C, int H, int W, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && C >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "attrib_step: bad shape N=%d C=%d H=%d W=%d", N, C,
             H, W);
  UD_REQUIRE(method == UD_ATTRIB_IG || method == UD_ATTRIB_SMOOTHGRAD, UD_ERR_INVALID,
             "attrib_step: unknown method %d (UD_ATTRIB_IG=0, UD_ATTRIB_SMOOTHGRAD=1)", method);
  UD_REQUIRE(steps >= 1, UD_ERR_INVALID, "attrib_step: steps=%d < 1 (the number of path points)", steps);
  UD_REQUIRE(N <= 65535, UD_ERR_UNSUPPORTED, "attrib_step: N=%d > 65535", N);
  const long long HW = (long long)H * W, P = HW * C;
  UD_REQUIRE(P <= (1LL << 31), UD_ERR_UNSUPPORTED, "attrib_step: %lld elements per sample > 2^31", P);
  UD_REQUIRE(x && acc && p && attr && map && k, UD_ERR_INVALID, "attrib_step: null pointer");
  UD_REQUIRE(alpha && w, UD_ERR_INVALID, "attrib_step: null step table (alpha, w)");
  UD_REQUIRE(method != UD_ATTRIB_SMOOTHGRAD || (sigma && seed), UD_ERR_INVALID,
             "attrib_step: SmoothGrad needs sigma and seed");
  UD_REQUIRE(p != x && p != g && p != acc && attr != acc, UD_ERR_INVALID, "attrib_step: p / attr alias an input");

  ExArgs a;
  a.x = x; a.b = base; a.g = g; a.acc = acc; a.p = p; a.attr = attr; a.map = map; a.k = k; a.alpha = alpha; a.w = w;
  a.sigma = sigma; a.ids = ids; a.seed = seed; a.bval = base_value; a.P = P; a.HW = HW; a.C = C; a.S = steps;
  a.chunks = ud_cdiv(P, EX_CHUNK);
  // float4 groups need every tensor at the same offset from a 16-byte boundary: true for torch allocations
  const uintptr_t al = (uintptr_t)x | (uintptr_t)(base ? base : x) | (uintptr_t)(g ? g : x) | (uintptr_t)acc |
                       (uintptr_t)p | (uintptr_t)attr;
  if ((al & 15) == 0) {
    ex_launch<true>(a, method, N, stream);
  } else {
    ex_launch<false>(a, method, N, stream);
  }
  int rc = ud_check_launch("attrib_step");
  if (rc || !g) return rc;
  ex_map_kernel<<<dim3(ud_cdiv(HW, EX_THREADS), N), EX_THREADS, 0, stream>>>(a);
  return ud_check_launch("attrib_step (map)");
}

// y[n, c, pix] = baseline where (rank[n, pix] < t[j]) != insertion, else x
__global__ void __launch_bounds__(EX_THREADS) ex_mask_kernel(const float* __restrict__ x, const float* __restrict__ b,
                                                            float bval, const int* __restrict__ rank, const int* t,
                                                            const int* jp, int points, float* __restrict__ y,
                                                            bool insertion, int C, long long HW) {
  const int j = *jp;
  if (j < 0 || j > points) return;
  const long long pix = (long long)blockIdx.x * EX_THREADS + threadIdx.x;
  if (pix >= HW) return;
  const int n = blockIdx.y;
  const bool use_b = (__ldg(rank + (long long)n * HW + pix) < __ldg(t + j)) != insertion;
  const long long o = (long long)n * C * HW + pix;
  for (int c = 0; c < C; ++c) {
    const long long i = o + (long long)c * HW;
    y[i] = use_b ? (b ? __ldg(b + i) : bval) : __ldg(x + i);
  }
}

extern "C" int ud_attrib_mask(const float* x, const float* base, float base_value, const int* rank, const int* t,
                              const int* j, int points, float* y, int insertion, int N, int C, int H, int W,
                              cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && C >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "attrib_mask: bad shape N=%d C=%d H=%d W=%d", N, C,
             H, W);
  UD_REQUIRE(insertion == 0 || insertion == 1, UD_ERR_INVALID, "attrib_mask: insertion must be 0 or 1, got %d",
             insertion);
  UD_REQUIRE(points >= 1, UD_ERR_INVALID, "attrib_mask: points=%d < 1", points);
  UD_REQUIRE(N <= 65535, UD_ERR_UNSUPPORTED, "attrib_mask: N=%d > 65535", N);
  const long long HW = (long long)H * W;
  UD_REQUIRE(HW <= (1LL << 30), UD_ERR_UNSUPPORTED, "attrib_mask: H*W=%lld > 2^30", HW);
  UD_REQUIRE(x && rank && t && j && y, UD_ERR_INVALID, "attrib_mask: null pointer");
  UD_REQUIRE(y != x && y != base, UD_ERR_INVALID, "attrib_mask: y aliases x or the baseline");
  ex_mask_kernel<<<dim3(ud_cdiv(HW, EX_THREADS), N), EX_THREADS, 0, stream>>>(x, base, base_value, rank, t, j, points,
                                                                              y, insertion != 0, C, HW);
  return ud_check_launch("attrib_mask");
}
