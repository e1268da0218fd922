// a5 / a6 -- dynamic filters: BatchNorm statistics and the fused mask stage   (SURVEY.md §8a rows a5, a6)
//
// Reference: FrequencyDynamicFilter.forward (model/modules.py:91-105) and
// SpatialDynamicFilter.forward (model/modules.py:120-134):
//     proj = act(BN(conv(x)))                      -- conv is the dense projection (library GEMM / tcgen05)
//     pre  = cat[mean_c proj, max_c proj, diff]    -- 2 + D channels
//     mask = sigmoid(conv1x1_{(2+D)->1}(pre));  out = mask * x
// Everything after the conv is fused here: BN-apply + activation + channel mean/max(+argmax) +
// 1x1 conv + sigmoid + mask*x read `proj` and `x` once and write `out` once; `proj` after BN/act
// is never materialised.  BN batch statistics are separate per-channel kernels because under
// DDP the engines convert these BNs to SyncBatchNorm (engine/forgery_engine.py:142) and the
// (mean, M2, count) triple must cross ranks between "stats" and "apply".
//
// Layout: NCHW fp32; a CTA owns one sample x 32 consecutive positions, 8 channel groups x 32
// lanes, so every global access is a coalesced 128-byte row segment.
#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

#define DF_MAX_PRE 16  // 2 + D
#define DF_GROUPS 32   // channel groups per CTA of the mask kernels (x 32 positions = 1024 threads): the channel loop of a
                       // thread is Cp/32 independent 128-byte row loads, all in flight at once

// ---------------------------------------------------------------- BN statistics (two-pass, per channel)
__global__ void __launch_bounds__(128)
df_bn_stats_kernel(const float* __restrict__ x, float* __restrict__ mean, float* __restrict__ m2, int N, int C,
                   int HW) {
  __shared__ float red[33];
  const int c = blockIdx.x;
  const int cnt = N * HW;
  float s = 0.f;
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    const int n = i / HW, p = i - n * HW;
    s += x[((long long)n * C + c) * HW + p];
  }
  const float mu = ud_block_sum(s, red) / (float)cnt;
  float q = 0.f;
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    const int n = i / HW, p = i - n * HW;
    const float d = x[((long long)n * C + c) * HW + p] - mu;
    q = fmaf(d, d, q);
  }
  q = ud_block_sum(q, red);
  if (threadIdx.x == 0) {
    mean[c] = mu;
    m2[c] = q;
  }
}

extern "C" int ud_bn_stats(const float* x, float* mean, float* m2, int N, int C, int HW, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && C >= 1 && HW >= 1, UD_ERR_INVALID, "bn_stats: bad shape N=%d C=%d HW=%d", N, C, HW);
  UD_REQUIRE(x && mean && m2, UD_ERR_INVALID, "bn_stats: null pointer");
  df_bn_stats_kernel<<<C, 128, 0, stream>>>(x, mean, m2, N, C, HW);
  return ud_check_launch("bn_stats");
}

// sum_dz[c] = sum dz, sum_dz_xh[c] = sum dz * xh, xh = (x - mean) * rstd
__global__ void __launch_bounds__(128)
df_bn_bwd_reduce_kernel(const float* __restrict__ dz, const float* __restrict__ x, const float* __restrict__ mean,
                        const float* __restrict__ rstd, float* __restrict__ sum_dz, float* __restrict__ sum_dz_xh,
                        int N, int C, int HW) {
  __shared__ float red[33];
  const int c = blockIdx.x;
  const int cnt = N * HW;
  const float mu = mean[c], rs = rstd[c];
  float a = 0.f, b = 0.f;
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    const int n = i / HW, p = i - n * HW;
    const long long idx = ((long long)n * C + c) * HW + p;
    const float g = dz[idx];
    a += g;
    b = fmaf(g, (x[idx] - mu) * rs, b);
  }
  a = ud_block_sum(a, red);
  b = ud_block_sum(b, red);
  if (threadIdx.x == 0) {
    sum_dz[c] = a;
    sum_dz_xh[c] = b;
  }
}

extern "C" int ud_bn_bwd_reduce(const float* dz, const float* x, const float* mean, const float* rstd, float* sum_dz,
                                float* sum_dz_xh, int N, int C, int HW, cudaStream_t stream) {
  UD_REQUIRE(N >= 1 && C >= 1 && HW >= 1, UD_ERR_INVALID, "bn_bwd_reduce: bad shape");
  UD_REQUIRE(dz && x && mean && rstd && sum_dz && sum_dz_xh, UD_ERR_INVALID, "bn_bwd_reduce: null pointer");
  df_bn_bwd_reduce_kernel<<<C, 128, 0, stream>>>(dz, x, mean, rstd, sum_dz, sum_dz_xh, N, C, HW);
  return ud_check_launch("bn_bwd_reduce");
}

// training: gx = gamma*rstd*(dz - sum_dz*inv_count - xh*sum_dz_xh*inv_count); eval (inv_count==0): gamma*rstd*dz
__global__ void df_bn_bwd_apply_kernel(const float* __restrict__ dz, const float* __restrict__ x,
                                       const float* __restrict__ mean, const float* __restrict__ rstd,
                                       const float* __restrict__ gamma, const float* __restrict__ sum_dz,
                                       const float* __restrict__ sum_dz_xh, float inv_count, float* __restrict__ gx,
                                       long long total, int C, int HW) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)((i / HW) % C);
    const float rs = rstd[c];
    const float k = (gamma ? gamma[c] : 1.f) * rs;
    float g = dz[i];
    if (inv_count != 0.f) {
      const float xh = (x[i] - mean[c]) * rs;
      g = g - sum_dz[c] * inv_count - xh * (sum_dz_xh[c] * inv_count);
    }
    gx[i] = k * g;
  }
}

extern "C" int ud_bn_bwd_apply(const float* dz, const float* x, const float* mean, const float* rstd,
                               const float* gamma, const float* sum_dz, const float* sum_dz_xh, float inv_count,
                               float* gx, int N, int C, int HW, cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && C >= 1 && HW >= 1, UD_ERR_INVALID, "bn_bwd_apply: bad shape");
  const long long total = (long long)N * C * HW;
  if (total == 0) return UD_OK;
  UD_REQUIRE(dz && x && mean && rstd && gx, UD_ERR_INVALID, "bn_bwd_apply: null pointer");
  UD_REQUIRE(inv_count == 0.f || (sum_dz && sum_dz_xh), UD_ERR_INVALID, "bn_bwd_apply: sums required in training");
  const int blocks = (int)min((long long)UD_NUM_SMS * 8, (total + 255) / 256);
  df_bn_bwd_apply_kernel<<<blocks, 256, 0, stream>>>(dz, x, mean, rstd, gamma, sum_dz, sum_dz_xh, inv_count, gx, total,
                                                     C, HW);
  return ud_check_launch("bn_bwd_apply");
}

// ---------------------------------------------------------------- fused mask stage, forward
__global__ void __launch_bounds__(DF_GROUPS * 32)
df_mask_fwd_kernel(const float* __restrict__ proj, const float* __restrict__ bn_mean, const float* __restrict__ bn_rstd,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ diff,
                   const float* __restrict__ w2, const float* __restrict__ x, float* __restrict__ mask,
                   float* __restrict__ out, float* __restrict__ pmean, float* __restrict__ pmax,
                   int* __restrict__ argmax, int Cp, int D, int Cx, int HW, int tiles, int act) {
  __shared__ float s_sum[DF_GROUPS][33];
  __shared__ float s_max[DF_GROUPS][33];
  __shared__ int s_arg[DF_GROUPS][33];
  __shared__ float s_mask[32];
  const int n = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int pos = tile * 32 + lane;
  const bool live = pos < HW;
  float sum = 0.f, mx = -INFINITY;
  int am = 0x7fffffff;
  if (live) {
    const float* pp = proj + (long long)n * Cp * HW + pos;
#pragma unroll 4
    for (int c = grp; c < Cp; c += DF_GROUPS) {
      const float rs = __ldg(bn_rstd + c);
      const float a = (gamma ? __ldg(gamma + c) : 1.f) * rs;
      const float b = (beta ? __ldg(beta + c) : 0.f) - __ldg(bn_mean + c) * a;
      const float v = ud_act_fwd(fmaf(pp[(long long)c * HW], a, b), act);
      sum += v;
      if (v > mx) {  // strict: first index wins inside a group (c increases)
        mx = v;
        am = c;
      }
    }
  }
  s_sum[grp][lane] = sum;
  s_max[grp][lane] = mx;
  s_arg[grp][lane] = am;
  __syncthreads();
  if (grp == 0) {
    float t = 0.f, m = -INFINITY;
    int a = 0x7fffffff;
#pragma unroll
    for (int q = 0; q < DF_GROUPS; ++q) {
      t += s_sum[q][lane];
      const float v = s_max[q][lane];
      const int ai = s_arg[q][lane];
      if (v > m || (v == m && ai < a)) {  // torch.max: first occurrence on ties
        m = v;
        a = ai;
      }
    }
    float mk = 0.f;
    if (live) {
      const float mean_c = t / (float)Cp;
      float s = __ldg(w2 + 0) * mean_c + __ldg(w2 + 1) * m;
      for (int d = 0; d < D; ++d) s = fmaf(__ldg(w2 + 2 + d), diff[((long long)n * D + d) * HW + pos], s);
      mk = ud_sigmoid(s);
      const long long o = (long long)n * HW + pos;
      mask[o] = mk;
      pmean[o] = mean_c;
      pmax[o] = m;
      argmax[o] = a;
    }
    s_mask[lane] = mk;
  }
  __syncthreads();
  if (out != nullptr && live) {
    const float mk = s_mask[lane];
    const long long base = (long long)n * Cx * HW + pos;
#pragma unroll 4
    for (int c = grp; c < Cx; c += DF_GROUPS) out[base + (long long)c * HW] = mk * x[base + (long long)c * HW];
  }
}

extern "C" int ud_dyfi_mask_fwd(const float* proj, const float* bn_mean, const float* bn_rstd, const float* gamma,
                                const float* beta, const float* diff, const float* w2, const float* x, float* mask,
                                float* out, float* pmean, float* pmax, int* argmax, int N, int Cp, int D, int Cx,
                                int HW, int act, cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && Cp >= 1 && D >= 0 && Cx >= 1 && HW >= 1 && 2 + D <= DF_MAX_PRE, UD_ERR_INVALID,
             "dyfi_mask_fwd: bad shape N=%d Cp=%d D=%d Cx=%d HW=%d", N, Cp, D, Cx, HW);
  if (N == 0) return UD_OK;
  UD_REQUIRE(proj && bn_mean && bn_rstd && w2 && mask && pmean && pmax && argmax && (D == 0 || diff) && (!out || x),
             UD_ERR_INVALID, "dyfi_mask_fwd: null pointer");
  const int tiles = ud_cdiv(HW, 32);
  df_mask_fwd_kernel<<<N * tiles, DF_GROUPS * 32, 0, stream>>>(proj, bn_mean, bn_rstd, gamma, beta, diff, w2, x, mask, out, pmean,
                                                    pmax, argmax, Cp, D, Cx, HW, tiles, act);
  return ud_check_launch("dyfi_mask_fwd");
}

// ---------------------------------------------------------------- fused mask stage, backward
// d_s = (g_mask + sum_c g_out*x) * m(1-m);  g_x = m*g_out;  g_w2[i] = sum d_s*pre_i;
// dz[c] = d_s * (w2[0]/Cp + [c==argmax] w2[1]) * act'(z_c)      (grad w.r.t. the BN output)
// GD: also g_diff[n,k,p] = w2[2+k] * d_s (the guide maps' gradient; nullable).  GD = false is the training path.
template <bool GD>
__global__ void __launch_bounds__(DF_GROUPS * 32)
df_mask_bwd_kernel(const float* __restrict__ proj, const float* __restrict__ bn_mean, const float* __restrict__ bn_rstd,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ diff,
                   const float* __restrict__ w2, const float* __restrict__ x, const float* __restrict__ mask,
                   const float* __restrict__ pmean, const float* __restrict__ pmax, const int* __restrict__ argmax,
                   const float* __restrict__ g_mask, const float* __restrict__ g_out, float* __restrict__ g_x,
                   float* __restrict__ dz, float* __restrict__ w2_part, float* __restrict__ g_diff, int Cp, int D,
                   int Cx, int HW, int tiles, int act) {
  __shared__ float s_t[DF_GROUPS][33];
  __shared__ float s_ds[32];
  const int n = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int pos = tile * 32 + lane;
  const bool live = pos < HW;
  const long long o = (long long)n * HW + pos;
  const float mk = live ? mask[o] : 0.f;
  float t = 0.f;
  if (g_out != nullptr && live) {
    const long long base = (long long)n * Cx * HW + pos;
#pragma unroll 4
    for (int c = grp; c < Cx; c += DF_GROUPS) {
      const float g = g_out[base + (long long)c * HW];
      t = fmaf(g, x[base + (long long)c * HW], t);
      g_x[base + (long long)c * HW] = mk * g;
    }
  }
  s_t[grp][lane] = t;
  __syncthreads();
  if (grp == 0) {
    float tt = 0.f;
#pragma unroll
    for (int q = 0; q < DF_GROUPS; ++q) tt += s_t[q][lane];
    const float gm = (g_mask != nullptr && live) ? g_mask[o] : 0.f;
    s_ds[lane] = live ? (gm + tt) * mk * (1.f - mk) : 0.f;
  }
  __syncthreads();
  const float ds = s_ds[lane];
  if (live) {
    const float wmean = __ldg(w2 + 0) / (float)Cp, wmax = __ldg(w2 + 1);
    const int am = argmax[o];
    const float* pp = proj + (long long)n * Cp * HW + pos;
    float* dzp = dz + (long long)n * Cp * HW + pos;
#pragma unroll 4
    for (int c = grp; c < Cp; c += DF_GROUPS) {
      const float rs = __ldg(bn_rstd + c);
      const float a = (gamma ? __ldg(gamma + c) : 1.f) * rs;
      const float b = (beta ? __ldg(beta + c) : 0.f) - __ldg(bn_mean + c) * a;
      const float z = fmaf(pp[(long long)c * HW], a, b);
      dzp[(long long)c * HW] = ds * (wmean + (c == am ? wmax : 0.f)) * ud_act_grad(z, act);
    }
  }
  // g_w2 partials (deterministic): index 0 mean, 1 max, 2.. diff
  if (grp == 0) {                       // only the 32 positions of the tile contribute: one warp, no block barrier
    for (int i = 0; i < 2 + D; ++i) {
      float v = 0.f;
      if (live) {
        const float pre = (i == 0) ? pmean[o] : (i == 1) ? pmax[o] : diff[((long long)n * D + (i - 2)) * HW + pos];
        v = ds * pre;
      }
      v = ud_warp_sum(v);
      if (lane == 0) w2_part[(long long)blockIdx.x * DF_MAX_PRE + i] = v;
    }
    if (GD && g_diff != nullptr && live) {
      for (int k = 0; k < D; ++k) g_diff[((long long)n * D + k) * HW + pos] = __ldg(w2 + 2 + k) * ds;
    }
  }
}

__global__ void df_w2_reduce_kernel(const float* __restrict__ part, float* __restrict__ g_w2, int nblocks, int npre) {
  __shared__ float red[33];
  const int i = blockIdx.x;
  float a = 0.f;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) a += part[(long long)b * DF_MAX_PRE + i];
  a = ud_block_sum(a, red);
  if (threadIdx.x == 0 && i < npre) g_w2[i] = a;
}

extern "C" size_t ud_dyfi_mask_bwd_workspace_bytes(int N, int HW) {
  return sizeof(float) * (size_t)N * ud_cdiv(HW, 32) * DF_MAX_PRE;
}

extern "C" int ud_dyfi_mask_bwd(const float* proj, const float* bn_mean, const float* bn_rstd, const float* gamma,
                                const float* beta, const float* diff, const float* w2, const float* x,
                                const float* mask, const float* pmean, const float* pmax, const int* argmax,
                                const float* g_mask, const float* g_out, float* g_x, float* dz, float* g_w2, float* g_diff,
                                void* ws, size_t ws_bytes, int N, int Cp, int D, int Cx, int HW, int act,
                                cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && Cp >= 1 && D >= 0 && Cx >= 1 && HW >= 1 && 2 + D <= DF_MAX_PRE, UD_ERR_INVALID,
             "dyfi_mask_bwd: bad shape");
  UD_REQUIRE(g_w2, UD_ERR_INVALID, "dyfi_mask_bwd: null pointer");
  if (N == 0) {
    UD_CUDA(cudaMemsetAsync(g_w2, 0, sizeof(float) * (2 + D), stream));
    return UD_OK;
  }
  UD_REQUIRE(proj && bn_mean && bn_rstd && w2 && mask && pmean && pmax && argmax && dz && ws && (D == 0 || diff) &&
                 (!g_out || (x && g_x)),
             UD_ERR_INVALID, "dyfi_mask_bwd: null pointer");
  UD_REQUIRE(ws_bytes >= ud_dyfi_mask_bwd_workspace_bytes(N, HW), UD_ERR_WORKSPACE, "dyfi_mask_bwd: workspace too small");
  if (D == 0) g_diff = nullptr;
  const int tiles = ud_cdiv(HW, 32);
  float* part = static_cast<float*>(ws);
  auto k = g_diff ? df_mask_bwd_kernel<true> : df_mask_bwd_kernel<false>;
  k<<<N * tiles, DF_GROUPS * 32, 0, stream>>>(proj, bn_mean, bn_rstd, gamma, beta, diff, w2, x, mask, pmean, pmax, argmax,
                                              g_mask, g_out, g_x, dz, part, g_diff, Cp, D, Cx, HW, tiles, act);
  int rc = ud_check_launch("dyfi_mask_bwd");
  if (rc != UD_OK) return rc;
  df_w2_reduce_kernel<<<2 + D, 128, 0, stream>>>(part, g_w2, N * tiles, 2 + D);
  return ud_check_launch("dyfi_w2_reduce");
}
