// a14 -- SpatialStyleTransfer: exact histogram (rank) matching, no grad               (SURVEY.md §8a row a14)
//
// Reference: model/modules.py:59-76
//     _, index_content = sort(content.view(B,C,-1));  value_style, _ = sort(style.view(B,C,-1))
//     inverse_index = index_content.argsort(-1)
//     out = content + (1-lmda) * value_style.gather(-1, inverse_index) - (1-lmda) * content       lmda [B] in [0.5,1)
// i.e. the pixel of rank r in the content plane takes (a blend with) the style plane's r-th smallest value.
// The reference runs two full sorts, an argsort and a gather per call (3 segmented CUB sorts on the GPU).
//
// Here: ONE CTA per (b, c) plane runs a stable least-significant-digit radix sort (4 passes of 8 bits over the
// order-preserving integer image of the floats) entirely through an L2-resident per-plane workspace:
//   * all four digit histograms come from one read of the plane (a histogram does not depend on the order);
//   * a pass walks the plane in tiles of 8192 keys; a warp owns 256 consecutive keys, ranks equal digits with
//     __match_any_sync (stable: item-major, lane-minor), one shared-memory counter per (warp, digit); 256 threads
//     turn the 32 per-warp counters of each digit into offsets; the scatter adds the running per-digit base;
//   * launch 1 sorts the STYLE planes (keys only) and stores the sorted values;
//   * launch 2 sorts the CONTENT planes carrying the pixel index; its last pass does not store the sorted order at
//     all: the key arriving at rank r belongs to pixel idx, so out[idx] = blend(content value, style_sorted[r]) is
//     written right there -- no argsort, no gather, no re-read of the content.
// Ties: equal content values keep their pixel order (stable); torch.sort leaves the order of ties unspecified, so the
// reference's own output is implementation-defined there (and only there).
//
// A third mode ranks attribution maps for the deletion / insertion faithfulness curves (ud_rank_desc): the keys are
// inverted (descending order), NaN keys sort after every number and -0 is keyed as +0, the pixel index is carried as in
// the content sort, and the last pass writes rank[idx] = r.
#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

#define SS_THREADS 1024
#define SS_WARPS (SS_THREADS / 32)
#define SS_ITEMS 8
#define SS_TILE (SS_THREADS * SS_ITEMS)

__device__ __forceinline__ uint32_t ss_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float ss_unkey(uint32_t k) {
  return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu));
}

#define SS_STYLE 0     // keys only, sorted values out
#define SS_CONTENT 1   // keys + pixel index, blend with the sorted style values out
#define SS_RANK 2      // descending keys + pixel index, int32 rank per pixel out

template <int MODE>
__device__ __forceinline__ uint32_t ss_mode_key(float f) {
  if (MODE != SS_RANK) return ss_key(f);
  return f != f ? 0xffffffffu : ~ss_key(f == 0.f ? 0.f : f);
}

// shared: hist[4][256] | tbase[256] | dbase[256] | whist[SS_WARPS][256]
template <int MODE>
__global__ void __launch_bounds__(SS_THREADS, 1)
ss_sort_kernel(const float* __restrict__ src, uint32_t* __restrict__ ws, const float* __restrict__ style_sorted,
               const float* __restrict__ lmda, void* __restrict__ dst, int E, int C) {
  __shared__ int hist[4][256];
  __shared__ int tbase[256];
  __shared__ int dbase[256];
  __shared__ int whist[SS_WARPS][256];
  constexpr bool IDX = MODE != SS_STYLE;      // carries the pixel index
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long seg = blockIdx.x;
  const float* sp = src + seg * (long long)E;
  // per-plane workspace: keys ping | keys pong (| idx ping | idx pong)
  uint32_t* wsp = ws + seg * (long long)E * (IDX ? 4 : 2);
  uint32_t* kbuf[2] = {wsp, wsp + E};
  uint32_t* ibuf[2] = {wsp + 2 * (long long)E, wsp + 3 * (long long)E};
  const uint32_t lt_mask = (1u << lane) - 1u;

  for (int i = tid; i < 4 * 256; i += SS_THREADS) (&hist[0][0])[i] = 0;
  __syncthreads();
  for (int i = tid; i < E; i += SS_THREADS) {
    const uint32_t k = ss_mode_key<MODE>(__ldg(sp + i));
    atomicAdd(&hist[0][k & 255], 1);
    atomicAdd(&hist[1][(k >> 8) & 255], 1);
    atomicAdd(&hist[2][(k >> 16) & 255], 1);
    atomicAdd(&hist[3][k >> 24], 1);
  }
  __syncthreads();

  float one_m_l = 0.f;
  const float* ssp = nullptr;
  float* op = static_cast<float*>(dst) + seg * (long long)E;
  if (MODE == SS_CONTENT) {
    one_m_l = 1.f - __ldg(lmda + seg / C);
    ssp = style_sorted + seg * (long long)E;
  }

#pragma unroll 1
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 8 * pass;
    // exclusive prefix of this pass's digit histogram -> running base per digit
    if (warp == 0) {
      int v[8], s = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = hist[pass][lane * 8 + j];
        s += v[j];
      }
      int incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      int run = incl - s;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        dbase[lane * 8 + j] = run;
        run += v[j];
      }
    }
    const uint32_t* kin = kbuf[(pass + 1) & 1];       // pass 0 reads src; passes 1..3 read what the previous one wrote
    const uint32_t* iin = ibuf[(pass + 1) & 1];
    uint32_t* kout = kbuf[pass & 1];
    uint32_t* iout = ibuf[pass & 1];
    __syncthreads();
#pragma unroll 1
    for (int t0 = 0; t0 < E; t0 += SS_TILE) {
      for (int i = tid; i < SS_WARPS * 256; i += SS_THREADS) (&whist[0][0])[i] = 0;
      __syncthreads();
      uint32_t key[SS_ITEMS], id[SS_ITEMS];
      int lr[SS_ITEMS];
      const int wbase = t0 + warp * (32 * SS_ITEMS);
#pragma unroll
      for (int j = 0; j < SS_ITEMS; ++j) {
        const int i = wbase + j * 32 + lane;
        key[j] = 0;
        id[j] = (uint32_t)i;
        if (i < E) {
          key[j] = (pass == 0) ? ss_mode_key<MODE>(__ldg(sp + i)) : kin[i];
          if (IDX && pass > 0) id[j] = iin[i];
        }
      }
#pragma unroll
      for (int j = 0; j < SS_ITEMS; ++j) {
        const int i = wbase + j * 32 + lane;
        const bool valid = i < E;
        const int d = valid ? (int)((key[j] >> shift) & 255u) : 256 + lane;       // invalid items match nobody
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const int before = __popc(peers & lt_mask);
        int old = 0;
        if (valid) old = whist[warp][d];
        __syncwarp();
        if (valid && before == 0) whist[warp][d] = old + __popc(peers);
        __syncwarp();
        lr[j] = old + before;
      }
      __syncthreads();
      if (tid < 256) {
        int run = 0;
#pragma unroll 8
        for (int w = 0; w < SS_WARPS; ++w) {
          const int v = whist[w][tid];
          whist[w][tid] = run;
          run += v;
        }
        const int b = dbase[tid];
        tbase[tid] = b;
        dbase[tid] = b + run;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < SS_ITEMS; ++j) {
        const int i = wbase + j * 32 + lane;
        if (i < E) {
          const int d = (int)((key[j] >> shift) & 255u);
          const int pos = tbase[d] + whist[warp][d] + lr[j];
          if (pass < 3) {
            kout[pos] = key[j];
            if (IDX) iout[pos] = id[j];
          } else if (MODE == SS_RANK) {
            static_cast<int*>(dst)[seg * (long long)E + id[j]] = pos;
          } else if (MODE == SS_CONTENT) {
            // the content pixel id[j] has rank pos:  content + (1-l)*matched - (1-l)*content, in the reference's order
            const float cv = ss_unkey(key[j]);
            const float mv = __ldg(ssp + pos);
            // (explicitly rounded products and sums: no FMA contraction, bit-identical to the three ATen kernels)
            op[id[j]] = __fsub_rn(__fadd_rn(cv, __fmul_rn(one_m_l, mv)), __fmul_rn(one_m_l, cv));
          } else {
            op[pos] = ss_unkey(key[j]);
          }
        }
      }
      __syncthreads();
    }
    __threadfence_block();
  }
}

extern "C" size_t ud_spatial_style_workspace_bytes(int N, int C, int HW) {
  if (N <= 0 || C <= 0 || HW <= 0) return 0;
  // sorted style values [N*C*HW] floats + the larger (content) sort workspace: 4 words per element
  return sizeof(float) * (size_t)N * C * HW * 5;
}

extern "C" int ud_spatial_style_transfer(const float* content, const float* style, const float* lmda, float* out, void* ws,
                                         size_t ws_bytes, int N, int C, int HW, cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && C >= 1 && HW >= 1, UD_ERR_INVALID, "spatial_style: bad shape N=%d C=%d HW=%d", N, C, HW);
  if (N == 0) return UD_OK;
  UD_REQUIRE(content && style && lmda && out && ws, UD_ERR_INVALID, "spatial_style: null pointer");
  UD_REQUIRE(ws_bytes >= ud_spatial_style_workspace_bytes(N, C, HW), UD_ERR_WORKSPACE, "spatial_style: workspace too small");
  UD_REQUIRE((long long)N * C <= 0x7fffffffLL && HW <= (1 << 30), UD_ERR_UNSUPPORTED, "spatial_style: tensor too large");
  float* sorted = static_cast<float*>(ws);
  uint32_t* sortws = reinterpret_cast<uint32_t*>(sorted + (size_t)N * C * HW);
  const int segs = N * C;
  ss_sort_kernel<SS_STYLE><<<segs, SS_THREADS, 0, stream>>>(style, sortws, nullptr, nullptr, sorted, HW, C);
  int rc = ud_check_launch("spatial_style_sort_style");
  if (rc != UD_OK) return rc;
  ss_sort_kernel<SS_CONTENT><<<segs, SS_THREADS, 0, stream>>>(content, sortws, sorted, lmda, out, HW, C);
  return ud_check_launch("spatial_style_sort_content");
}

extern "C" size_t ud_rank_desc_workspace_bytes(int N, int HW) {
  if (N <= 0 || HW <= 0) return 0;
  return sizeof(uint32_t) * (size_t)N * HW * 4;   // keys and pixel indices, ping and pong
}

extern "C" int ud_rank_desc(const float* map, int* rank, int N, int HW, void* ws, size_t ws_bytes, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && HW >= 1, UD_ERR_INVALID, "rank_desc: bad shape N=%d HW=%d", N, HW);
  UD_REQUIRE(N <= 65535 && HW <= (1 << 30), UD_ERR_UNSUPPORTED, "rank_desc: N=%d > 65535 or HW=%d > 2^30", N, HW);
  UD_REQUIRE(map && rank, UD_ERR_INVALID, "rank_desc: null pointer");
  const size_t need = ud_rank_desc_workspace_bytes(N, HW);
  UD_REQUIRE(ws && ws_bytes >= need, UD_ERR_WORKSPACE, "rank_desc: workspace of %zu bytes, %zu needed", ws_bytes, need);
  ss_sort_kernel<SS_RANK><<<N, SS_THREADS, 0, stream>>>(map, static_cast<uint32_t*>(ws), nullptr, nullptr, rank, HW, 1);
  return ud_check_launch("rank_desc");
}
