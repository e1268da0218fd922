// a1 -- reconstruction-loss tail, forward and backward        (SURVEY.md §8a row a1)
//
// Reference: model/unidefense.py:244-253 (Eb4), :423-433 (Res18), :618-628 (Res50):
//     rec     = bilinear(dec -> HxW, align_corners=True)
//     spatial = mean_{c,h,w} |rec - x|
//     freq    = mean_{c,h,k} |Re dF| + |Im dF|,   dF = rfft2(rec) - rfft2(x)
// By linearity dF = rfft2(rec - x) (SURVEY App. B.1), so ONE 2-D real FFT of d = rec - x per
// plane is computed instead of two, and neither spectrum is ever written to HBM.
//
// Forward  = rows kernel (upsample + diff + |d| partial sums + packed real row FFTs -> Y)
//          + cols kernel (column FFTs of Y + |Re|+|Im| partial sums + sign bytes)
//          + finalize   (fixed-order sum of the partials -> spatial[n], freq[n]).
// Backward = cols-inverse kernel (sign spectrum -> inverse column FFTs -> T)
//          + rows-inverse kernel (Hermitian-folded packed inverse row FFTs + sign(d) term
//            + transposed bilinear into g_dec).
// Y/T is an L2-resident workspace holding `chunk` samples' half spectra [plane][H][WhP].
//
// HBM traffic per sample (fp32): fwd reads dec+x, writes rec (+1 B/bin signs);
// bwd reads dec+x(+signs), writes g_dec.
#include "../../include/unidefense_b200.h"

#include "ud_fft.cuh"
#include "ud_fft_any.cuh"

// second-generation kernels for the configured image sizes (ud_recon_tail2.cu)
bool ud_rt2_supported(int h, int w, int H, int W);
int ud_rt2_rows_lpc(void);
size_t ud_rt2_workspace_plane_bytes(int H, int W);
int ud_rt2_fwd(const float* dec, const float* x, float* rec, float2* Z, float* part_sp, float* part_fr, uint8_t* signs,
               int plane0, int planes, int h, int w, int H, int W, int row_tiles, int col_tiles, cudaStream_t stream);
int ud_rt2_bwd(const float* dec, const float* x, const uint8_t* signs, const float* g_spatial, const float* g_freq,
               float* g_dec, float* g_x, float2* T, int plane0, int planes, int C, int h, int w, int H, int W, int row_tiles,
               int col_tiles, float gscale, float sp_scale, cudaStream_t stream);
// Each rows-CTA of ud_recon_tail2.cu walks one step of ud_rt2_rows_lpc() (16) row pairs.  Measured at N=32, 380^2: one
// step per CTA (12 row tiles per plane, ~4 waves) and two (6 tiles, ~2 waves) take the same time (101 / 89 us fwd / bwd),
// three is 10-30 % slower: the kernels are bound per SM (issue + L2 latency at 20 resident warps), not by wave shape.
#define RT2_COLS_PER_TILE 16

#define RT_ROW_T 256   // threads of the rows kernels
#define RT_ROW_L 12    // row PAIRS (complex lines) per CTA of the rows kernels  -> 24 image rows
#define RT_COL_T 320   // threads of the cols kernels
#define RT_COL_L 16    // columns per CTA of the cols kernels (16 float2 = one 128-byte line per row)
// Lines longer than shared memory holds at those counts (long Bluestein lines, m = 1024 or 2048) run instantiations
// with a half or a quarter of them: rt_row_lines / rt_col_lines pick the largest that fits.
#define RT_HSTAGE 12   // rows_bwd: max horizontal-transpose items per thread kept in registers
#define RT_VGRP 3      // row pairs whose vertical lerps are staged per barrier (every row-pair count % RT_VGRP == 0)

static inline int rt_whp(int W) { return ((W / 2 + 1) + 15) & ~15; }  // padded half width (float2)

__device__ __forceinline__ void rt_tab(const float2 t, int in_size, int& i0, int& i1, float& l0, float& l1) {
  i0 = __float_as_int(t.x);
  i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  l1 = t.y;
  l0 = 1.f - l1;
}

// Vertical lerp of the two image rows (ra, ra+1) of a pair into vA/vB [w] (shared memory).
__device__ __forceinline__ void rt_vrows(const float* __restrict__ decp, const float2* __restrict__ ytab_g, int ra, int h,
                                         int w, int H, float* __restrict__ vA, float* __restrict__ vB) {
  if (ra >= H) return;
  int a0, a1, b0, b1;
  float la0, la1, lb0, lb1;
  rt_tab(__ldg(ytab_g + ra), h, a0, a1, la0, la1);
  const bool has_b = ra + 1 < H;
  rt_tab(__ldg(ytab_g + (has_b ? ra + 1 : ra)), h, b0, b1, lb0, lb1);
  const float* pa0 = decp + (long long)a0 * w;
  const float* pa1 = decp + (long long)a1 * w;
  const float* pb0 = decp + (long long)b0 * w;
  const float* pb1 = decp + (long long)b1 * w;
  for (int c = threadIdx.x; c < w; c += blockDim.x) {
    vA[c] = la0 * __ldg(pa0 + c) + la1 * __ldg(pa1 + c);
    vB[c] = has_b ? (lb0 * __ldg(pb0 + c) + lb1 * __ldg(pb1 + c)) : 0.f;
  }
}

// ------------------------------------------------------------------------------------------
// forward rows: grid (row_tiles, planes_in_chunk)
//   shared: tw[n] | xtab[n] | buf0[L*LS] (| buf1[L*LS] when the plan ping-pongs) | vbuf[2][2][w]
// ------------------------------------------------------------------------------------------
template <class Plan, int L>
__global__ void __launch_bounds__(RT_ROW_T)
rt_rows_fwd_kernel(Plan plan, const float* __restrict__ dec, const float* __restrict__ x,
                   float* __restrict__ rec, float2* __restrict__ Y, float* __restrict__ part_spatial,
                   const float2* __restrict__ tw_g, const float2* __restrict__ ytab_g,
                   const float2* __restrict__ xtab_g, int plane0, int h, int w, int H, int W, int row_tiles) {
  static_assert(L % RT_VGRP == 0, "row pairs are staged in groups of RT_VGRP");
  extern __shared__ float2 smem[];
  const int n = plan.n();  // == W
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* xtab = tw + m;
  float2* buf0 = xtab + n;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;
  float* vbuf = reinterpret_cast<float*>(buf1 + L * LS);
  __shared__ float red[33];

  const int tile = blockIdx.x;
  const int pl = blockIdx.y;             // plane within chunk
  const long long plane = plane0 + pl;   // global (n*C + c)
  const int r0 = tile * (2 * L);
  W = n;                                 // W == n: lets static plans constant-fold every index below
  const int Wh = n / 2 + 1;
  const int WhP = (Wh + 15) & ~15;

  for (int t = threadIdx.x; t < m; t += RT_ROW_T) tw[t] = __ldg(tw_g + t);
  for (int t = threadIdx.x; t < n; t += RT_ROW_T) xtab[t] = __ldg(xtab_g + t);
  const float* decp = dec + plane * (long long)h * w;
  const float* xp = x + plane * (long long)H * W;
  float* recp = rec + plane * (long long)H * W;

  // whole x tile in flight first: x[ra][c] -> line[p][c].x, x[ra+1][c] -> .y (overwritten in place by d below)
  for (int p = 0; p < L; ++p) {
    const int ra = r0 + 2 * p;
    if (ra >= H) break;
    const float* xa_p = xp + (long long)ra * W;
    float2* line = buf0 + p * LS;
    const bool has_b = ra + 1 < H;
    for (int c = threadIdx.x; c < W; c += RT_ROW_T) {
      ud_cp_async4(&line[c].x, xa_p + c);
      if (has_b) ud_cp_async4(&line[c].y, xa_p + W + c);
    }
  }
  ud_cp_async_commit();
  for (int q = 0; q < RT_VGRP; ++q) rt_vrows(decp, ytab_g, r0 + 2 * q, h, w, H, vbuf + 2 * q * w, vbuf + (2 * q + 1) * w);
  ud_cp_async_wait_all();
  __syncthreads();
  float acc = 0.f;
  for (int g = 0; g < L / RT_VGRP; ++g) {
    if (g + 1 < L / RT_VGRP) {
      float* nv = vbuf + ((g + 1) & 1) * (2 * RT_VGRP) * w;
      for (int q = 0; q < RT_VGRP; ++q)
        rt_vrows(decp, ytab_g, r0 + 2 * ((g + 1) * RT_VGRP + q), h, w, H, nv + 2 * q * w, nv + (2 * q + 1) * w);
    }
    const float* vg = vbuf + (g & 1) * (2 * RT_VGRP) * w;
#pragma unroll
    for (int q = 0; q < RT_VGRP; ++q) {
      const int p = g * RT_VGRP + q;
      const int ra = r0 + 2 * p;
      const float* vA = vg + 2 * q * w;
      const float* vB = vA + w;
      float2* line = buf0 + p * LS;
      if (ra >= H) {
        for (int c = threadIdx.x; c < W; c += RT_ROW_T) line[c] = make_float2(0.f, 0.f);
      } else {
        const bool has_b = ra + 1 < H;
        float* ra_p = recp + (long long)ra * W;
        for (int c = threadIdx.x; c < W; c += RT_ROW_T) {
          int i0, i1;
          float l0, l1;
          rt_tab(xtab[c], w, i0, i1, l0, l1);
          const float2 xv = line[c];
          const float va = l0 * vA[i0] + l1 * vA[i1];
          __stcs(ra_p + c, va);
          const float dA = va - xv.x;
          float dB = 0.f;
          if (has_b) {
            const float vb = l0 * vB[i0] + l1 * vB[i1];
            __stcs(ra_p + W + c, vb);
            dB = vb - xv.y;
          }
          acc += fabsf(dA) + fabsf(dB);
          line[c] = make_float2(dA, dB);
        }
      }
    }
    __syncthreads();
  }
  float2* res = plan.run(buf0, buf1, tw, L, LS);

  // unpack the two real rows of each pair: A[k] = (Z[k]+conj Z[n-k])/2, B[k] = (Z[k]-conj Z[n-k])/(2i)
  float2* Yp = Y + (long long)pl * H * WhP;
  for (int t = threadIdx.x; t < L * Wh; t += RT_ROW_T) {
    const int p = t / Wh, k = t - p * Wh;
    const int ra = r0 + 2 * p;
    if (ra >= H) continue;
    const float2 z = res[p * LS + k];
    const float2 zn = res[p * LS + (k == 0 ? 0 : n - k)];
    Yp[(long long)ra * WhP + k] = make_float2(0.5f * (z.x + zn.x), 0.5f * (z.y - zn.y));
    if (ra + 1 < H) Yp[(long long)(ra + 1) * WhP + k] = make_float2(0.5f * (z.y + zn.y), -0.5f * (z.x - zn.x));
  }
  const float tot = ud_block_sum(acc, red);
  if (threadIdx.x == 0) part_spatial[plane * row_tiles + tile] = tot;
}

// ------------------------------------------------------------------------------------------
// forward cols: grid (col_tiles, planes_in_chunk).  Column FFT length n = H.
// ------------------------------------------------------------------------------------------
template <class Plan, int L>
__global__ void __launch_bounds__(RT_COL_T)
rt_cols_fwd_kernel(Plan plan, const float2* __restrict__ Y, float* __restrict__ part_freq,
                   uint8_t* __restrict__ signs, const float2* __restrict__ tw_g, int plane0, int H, int W,
                   int col_tiles) {
  extern __shared__ float2 smem[];
  const int n = plan.n();  // == H
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* buf0 = tw + m;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;
  __shared__ float red[33];

  const int tile = blockIdx.x;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  H = n;                                 // H == n: constant-folds the index math for static plans
  const int Wh = W / 2 + 1;
  const int WhP = (Wh + 15) & ~15;
  const int k0 = tile * L;
  const int ncols = min(L, Wh - k0);

  for (int t = threadIdx.x; t < m; t += RT_COL_T) tw[t] = __ldg(tw_g + t);
  const float2* Yp = Y + (long long)pl * H * WhP;
  for (int t = threadIdx.x; t < H * L; t += RT_COL_T) {
    const int r = t / L, cc = t - r * L;
    if (cc < ncols) ud_cp_async8(&buf0[cc * LS + r], Yp + (long long)r * WhP + k0 + cc);
    else buf0[cc * LS + r] = make_float2(0.f, 0.f);
  }
  ud_cp_async_commit();
  ud_cp_async_wait_all();
  __syncthreads();
  float2* res = plan.run(buf0, buf1, tw, L, LS);

  float acc = 0.f;
  for (int t = threadIdx.x; t < ncols * H; t += RT_COL_T) {
    const int cc = t / H, j = t - cc * H;
    const float2 v = res[cc * LS + j];
    acc += fabsf(v.x) + fabsf(v.y);
    if (signs != nullptr) {
      const uint8_t sr = v.x > 0.f ? 1 : (v.x < 0.f ? 2 : 0);
      const uint8_t si = v.y > 0.f ? 1 : (v.y < 0.f ? 2 : 0);
      signs[(plane * Wh + (k0 + cc)) * (long long)H + j] = (uint8_t)(sr | (si << 2));
    }
  }
  const float tot = ud_block_sum(acc, red);
  if (threadIdx.x == 0) part_freq[plane * col_tiles + tile] = tot;
}

// fixed-order reduction of the partial sums: grid N, block 128
__global__ void rt_finalize_kernel(const float* __restrict__ part_spatial, const float* __restrict__ part_freq,
                                   float* __restrict__ spatial, float* __restrict__ freq, int C, int row_tiles,
                                   int col_tiles, float inv_sp, float inv_fr) {
  __shared__ float red[33];
  const int nsmp = blockIdx.x;
  float a = 0.f, b = 0.f;
  const int ns = C * row_tiles, nf = C * col_tiles;
  for (int i = threadIdx.x; i < ns; i += blockDim.x) a += part_spatial[(long long)nsmp * ns + i];
  for (int i = threadIdx.x; i < nf; i += blockDim.x) b += part_freq[(long long)nsmp * nf + i];
  a = ud_block_sum(a, red);
  b = ud_block_sum(b, red);
  if (threadIdx.x == 0) {
    spatial[nsmp] = a * inv_sp;
    freq[nsmp] = b * inv_fr;
  }
}

// ------------------------------------------------------------------------------------------
// backward cols (inverse column FFT of the sign spectrum): grid (col_tiles, planes_in_chunk)
// T[r,k] = sum_j S[j,k] e^{+2 pi i j r / H},  S = gf * (sgn Re D + i sgn Im D)
// inverse via the swap trick: IFFT(z) = swap(FFT(swap(z))).
// ------------------------------------------------------------------------------------------
template <class Plan, int L>
__global__ void __launch_bounds__(RT_COL_T)
rt_cols_bwd_kernel(Plan plan, const uint8_t* __restrict__ signs, const float* __restrict__ g_freq,
                   float2* __restrict__ T, const float2* __restrict__ tw_g, int plane0, int C, int H, int W,
                   float gscale) {
  extern __shared__ float2 smem[];
  const int n = plan.n();
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* buf0 = tw + m;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;

  const int tile = blockIdx.x;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int smp = (int)(plane / C);
  if (g_freq[smp] == 0.f) return;  // whole plane contributes nothing; the rows kernel skips its FFT too
  const float gf = g_freq[smp] * gscale;
  H = n;
  const int Wh = W / 2 + 1;
  const int WhP = (Wh + 15) & ~15;
  const int k0 = tile * L;
  const int ncols = min(L, Wh - k0);

  for (int t = threadIdx.x; t < m; t += RT_COL_T) tw[t] = __ldg(tw_g + t);
  for (int t = threadIdx.x; t < L * H; t += RT_COL_T) {
    const int cc = t / H, j = t - cc * H;
    float2 v = make_float2(0.f, 0.f);
    if (cc < ncols) {
      const uint8_t s = signs[(plane * Wh + (k0 + cc)) * (long long)H + j];
      const float sr = (s & 1) ? gf : ((s & 2) ? -gf : 0.f);
      const float si = (s & 4) ? gf : ((s & 8) ? -gf : 0.f);
      v = make_float2(si, sr);  // swapped
    }
    buf0[cc * LS + j] = v;
  }
  __syncthreads();
  float2* res = plan.run(buf0, buf1, tw, L, LS);
  float2* Tp = T + (long long)pl * H * WhP;
  for (int t = threadIdx.x; t < H * L; t += RT_COL_T) {
    const int r = t / L, cc = t - r * L;
    if (cc < ncols) {
      const float2 v = res[cc * LS + r];
      Tp[(long long)r * WhP + k0 + cc] = make_float2(v.y, v.x);  // swap back
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward rows: grid (row_tiles, planes_in_chunk).
// g_rec[r,c] = gs*sign(d[r,c]) + Re sum_{k<Wh} T[r,k] e^{+2 pi i k c / W}; then the transposed
// bilinear resize accumulates into g_dec (pre-zeroed).  Two rows are packed per complex line by
// folding T into its Hermitian part Th (Re IFFT(T) == IFFT(Th)) and transforming Th_a + i Th_b.
//   shared: tw[n] | xtab[n] | buf0[L*LS] (| buf1) | vbuf[2][2][w]
// After the FFT a line holds (g_b[c], g_a[c]) per column.  The transposed resize runs horizontally
// first (gather through xtab, both rows of a pair at once, results staged in registers and written back
// over the line), then vertically: one thread per dec column walks the tile's rows in order carrying two
// running sums (rows i and i+1) and flushes each finished dec row with one atomicAdd.
// GX: also g_x = -g_rec at full resolution from the finished lines (zeros for planes whose sample has gs == gf == 0);
// g_dec may then be NULL.  GX = false is the training path.
// ------------------------------------------------------------------------------------------
template <class Plan, bool GX, int L>
__global__ void __launch_bounds__(RT_ROW_T)
rt_rows_bwd_kernel(Plan plan, const float* __restrict__ dec, const float* __restrict__ x,
                   const float2* __restrict__ T, const float* __restrict__ g_spatial,
                   const float* __restrict__ g_freq, float* __restrict__ g_dec, float* __restrict__ g_x,
                   const float2* __restrict__ tw_g, const float2* __restrict__ ytab_g,
                   const float2* __restrict__ xtab_g, const int2* __restrict__ jtab_g, int plane0, int C, int h,
                   int w, int H, int W, float sp_scale) {
  static_assert(L % RT_VGRP == 0, "row pairs are staged in groups of RT_VGRP");
  extern __shared__ float2 smem[];
  const int n = plan.n();  // == W
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* xtab = tw + m;
  float2* buf0 = xtab + n;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;
  float* vbuf = reinterpret_cast<float*>(buf1 + L * LS);

  const int tile = blockIdx.x;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int smp = (int)(plane / C);
  const float gs = g_spatial[smp] * sp_scale;
  const bool has_f = g_freq[smp] != 0.f;
  const int r0 = tile * (2 * L);
  if (gs == 0.f && !has_f) {
    if (GX) {                            // the tile's rows of g_x are zero
      float* gxp = g_x + plane * (long long)H * n;
      const long long e = (long long)min(H, r0 + 2 * L) * n;
      for (long long i = (long long)r0 * n + threadIdx.x; i < e; i += RT_ROW_T) gxp[i] = 0.f;
    }
    return;
  }
  W = n;
  const int Wh = n / 2 + 1;
  const int WhP = (Wh + 15) & ~15;
  const int nrows = min(2 * L, H - r0);

  for (int t = threadIdx.x; t < m; t += RT_ROW_T) tw[t] = __ldg(tw_g + t);
  for (int t = threadIdx.x; t < n; t += RT_ROW_T) xtab[t] = __ldg(xtab_g + t);
  // sign(rec - x) of the tile first (2+2 bits per row pair and column), while the buffer is still free:
  // x is prefetched into the lines with cp.async exactly like the forward does.
  uint8_t* sgn = reinterpret_cast<uint8_t*>(vbuf + 4 * RT_VGRP * w);   // [L][n]
  if (gs != 0.f) {
    const float* decp = dec + plane * (long long)h * w;
    const float* xp = x + plane * (long long)H * W;
    for (int p = 0; p < L; ++p) {
      const int ra = r0 + 2 * p;
      if (ra >= H) break;
      const float* xa_p = xp + (long long)ra * W;
      float2* line = buf0 + p * LS;
      const bool has_b = ra + 1 < H;
      for (int c = threadIdx.x; c < W; c += RT_ROW_T) {
        ud_cp_async4(&line[c].x, xa_p + c);
        if (has_b) ud_cp_async4(&line[c].y, xa_p + W + c);
      }
    }
    ud_cp_async_commit();
    for (int q = 0; q < RT_VGRP; ++q) rt_vrows(decp, ytab_g, r0 + 2 * q, h, w, H, vbuf + 2 * q * w, vbuf + (2 * q + 1) * w);
    ud_cp_async_wait_all();
    __syncthreads();
    for (int g = 0; g < L / RT_VGRP; ++g) {
      if (g + 1 < L / RT_VGRP) {
        float* nv = vbuf + ((g + 1) & 1) * (2 * RT_VGRP) * w;
        for (int q = 0; q < RT_VGRP; ++q)
          rt_vrows(decp, ytab_g, r0 + 2 * ((g + 1) * RT_VGRP + q), h, w, H, nv + 2 * q * w, nv + (2 * q + 1) * w);
      }
      const float* vg = vbuf + (g & 1) * (2 * RT_VGRP) * w;
#pragma unroll
      for (int q = 0; q < RT_VGRP; ++q) {
        const int p = g * RT_VGRP + q;
        const int ra = r0 + 2 * p;
        const float* vA = vg + 2 * q * w;
        const float* vB = vA + w;
        const float2* line = buf0 + p * LS;
        const bool live = ra < H, has_b = ra + 1 < H;
        for (int c = threadIdx.x; c < W; c += RT_ROW_T) {
          uint8_t code = 0;
          if (live) {
            int i0, i1;
            float l0, l1;
            rt_tab(xtab[c], w, i0, i1, l0, l1);
            const float2 xv = line[c];
            const float dA = (l0 * vA[i0] + l1 * vA[i1]) - xv.x;
            code = dA > 0.f ? 1 : (dA < 0.f ? 2 : 0);
            if (has_b) {
              const float dB = (l0 * vB[i0] + l1 * vB[i1]) - xv.y;
              code |= dB > 0.f ? 4 : (dB < 0.f ? 8 : 0);
            }
          }
          sgn[p * n + c] = code;
        }
      }
      __syncthreads();
    }
  }

  float2* res = buf0;
  if (has_f) {
    const float2* Tp = T + (long long)pl * H * WhP;
    // build V = Th_a + i Th_b (swapped for the inverse) for k in [0, Wh) and its mirror n-k
    for (int t = threadIdx.x; t < L * Wh; t += RT_ROW_T) {
      const int p = t / Wh, k = t - p * Wh;
      const int ra = r0 + 2 * p;
      float2 ta = make_float2(0.f, 0.f), tb = make_float2(0.f, 0.f);
      if (ra < H) ta = Tp[(long long)ra * WhP + k];
      if (ra + 1 < H) tb = Tp[(long long)(ra + 1) * WhP + k];
      float2* line = buf0 + p * LS;
      const bool self_paired = (k == 0) || (2 * k == n);
      if (self_paired) {
        // Th = Re T ; V = (Re Ta, Re Tb) ; swapped -> (Re Tb, Re Ta)
        line[k] = make_float2(tb.x, ta.x);
      } else {
        const float ar = 0.5f * ta.x, ai = 0.5f * ta.y, br = 0.5f * tb.x, bi = 0.5f * tb.y;
        // V[k] = (ar - bi, ai + br) ; V[n-k] = (ar + bi, br - ai) ; store swapped
        line[k] = make_float2(ai + br, ar - bi);
        line[n - k] = make_float2(br - ai, ar + bi);
      }
    }
    __syncthreads();
    res = plan.run(buf0, buf1, tw, L, LS);   // res[p][c] = (g_b[c], g_a[c])
  } else {
    for (int t = threadIdx.x; t < L * LS; t += RT_ROW_T) buf0[t] = make_float2(0.f, 0.f);
    __syncthreads();
  }
  if (gs != 0.f) {  // g += gs * sign(rec - x)
    for (int t = threadIdx.x; t < L * n; t += RT_ROW_T) {
      const int p = t / n, c = t - p * n;
      const uint8_t code = sgn[t];
      float2 g = res[p * LS + c];
      g.y += (code & 1) ? gs : ((code & 2) ? -gs : 0.f);
      g.x += (code & 4) ? gs : ((code & 8) ? -gs : 0.f);
      res[p * LS + c] = g;
    }
    __syncthreads();
  }

  if (GX) {                              // g_x = -g_rec; res[p][c] = (g_b[c], g_a[c])
    float* gxp = g_x + (plane * H + r0) * (long long)n;
    for (int t = threadIdx.x; t < nrows * n; t += RT_ROW_T) {
      const int rr = t / n, c = t - rr * n;
      const float2 g2 = res[(rr >> 1) * LS + c];
      __stcs(gxp + t, (rr & 1) ? -g2.x : -g2.y);
    }
    if (g_dec == nullptr) return;        // g_x only: no transposed resize
  }
  float* gd = g_dec + plane * (long long)h * w;
  const int items = L * w;
  if (items <= RT_HSTAGE * RT_ROW_T && w <= n) {   // staged results are written back over the line (n slots)
    // horizontal transposed lerp, both rows of a pair per item, staged in registers.  jtab[j] = first/last
    // output column whose two taps include dec column j (exact, from the same fp32 table as the forward).
    float2 hv[RT_HSTAGE];
    int p = 0, j = threadIdx.x;
    while (j >= w) { j -= w; ++p; }
#pragma unroll
    for (int s = 0; s < RT_HSTAGE; ++s) {
      hv[s] = make_float2(0.f, 0.f);
      if (p < L) {
        const int2 cr = __ldg(jtab_g + j);
        const float2* line = res + p * LS;
        float ax = 0.f, ay = 0.f;
        for (int c = cr.x; c <= cr.y; ++c) {
          const float2 t = xtab[c];
          const int i0 = __float_as_int(t.x);
          const float wgt = (i0 == j) ? (1.f - t.y) + ((i0 == w - 1) ? t.y : 0.f) : t.y;   // i0 == j-1 -> the l1 tap
          const float2 g = line[c];
          ax = fmaf(wgt, g.x, ax);
          ay = fmaf(wgt, g.y, ay);
        }
        hv[s] = make_float2(ax, ay);
      }
      j += RT_ROW_T;
      while (j >= w) { j -= w; ++p; }
    }
    __syncthreads();
    p = 0;
    j = threadIdx.x;
    while (j >= w) { j -= w; ++p; }
#pragma unroll
    for (int s = 0; s < RT_HSTAGE; ++s) {
      if (p < L) res[p * LS + j] = hv[s];
      j += RT_ROW_T;
      while (j >= w) { j -= w; ++p; }
    }
    __syncthreads();
    // vertical transposed lerp: thread j walks the rows of the tile
    for (int j = threadIdx.x; j < w; j += RT_ROW_T) {
      int cur = __float_as_int(__ldg(ytab_g + r0).x);
      float acc0 = 0.f, acc1 = 0.f;
      for (int rr = 0; rr < nrows; ++rr) {
        int i0, i1;
        float l0, l1;
        rt_tab(__ldg(ytab_g + r0 + rr), h, i0, i1, l0, l1);
        while (cur < i0) {
          if (acc0 != 0.f) atomicAdd(gd + (long long)cur * w + j, acc0);
          acc0 = acc1;
          acc1 = 0.f;
          ++cur;
        }
        const float2 g2 = res[(rr >> 1) * LS + j];
        const float v = (rr & 1) ? g2.x : g2.y;
        acc0 = fmaf(l0, v, acc0);
        if (i1 > i0) acc1 = fmaf(l1, v, acc1);
        else acc0 = fmaf(l1, v, acc0);
      }
      if (acc0 != 0.f) atomicAdd(gd + (long long)cur * w + j, acc0);
      if (acc1 != 0.f && cur + 1 < h) atomicAdd(gd + (long long)(cur + 1) * w + j, acc1);
    }
  } else {
    // wide decoder planes: no register staging; distribute each horizontal result with two atomics
    for (int it = threadIdx.x; it < nrows * w; it += RT_ROW_T) {
      const int rr = it / w, j = it - rr * w;
      const int2 cr = __ldg(jtab_g + j);
      const float2* line = res + (rr >> 1) * LS;
      float a = 0.f;
      for (int c = cr.x; c <= cr.y; ++c) {
        int i0, i1;
        float l0, l1;
        rt_tab(xtab[c], w, i0, i1, l0, l1);
        const float wgt = ((i0 == j) ? l0 : 0.f) + ((i1 == j) ? l1 : 0.f);
        const float2 g = line[c];
        a = fmaf(wgt, (rr & 1) ? g.x : g.y, a);
      }
      int i0, i1;
      float l0, l1;
      rt_tab(__ldg(ytab_g + r0 + rr), h, i0, i1, l0, l1);
      if (a != 0.f) {
        atomicAdd(gd + (long long)i0 * w + j, l0 * a);
        if (l1 != 0.f) atomicAdd(gd + (long long)i1 * w + j, l1 * a);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// m: points per line buffer / staged twiddles (UdAnyPlan::m: n, or the Bluestein length for sizes with a prime factor
// > 23).  The plans are not in place, so the kernels keep two line buffers of L lines each.
static size_t rt_rows_fixed_smem(int n, int m, int w) {   // tw[m] | xtab[n] | vbuf
  return sizeof(float2) * ((size_t)m + n) + sizeof(float) * 4ull * RT_VGRP * w;
}
static size_t rt_rows_smem(int n, int m, int w, int L) {
  return rt_rows_fixed_smem(n, m, w) + sizeof(float2) * 2ull * L * (size_t)(m | 1) +
         (size_t)L * n;   // + sign bytes of the tile (rows_bwd)
}
static size_t rt_cols_smem(int m, int L) {
  return sizeof(float2) * ((size_t)m + 2ull * L * (size_t)(m | 1));
}
// Static shared memory of rt_rows_fwd_kernel / rt_cols_fwd_kernel: red[33] as ptxas lays it out.  The per-CTA limit
// holds static and dynamic bytes together, so the line counts below leave room for it.
#define RT_STATIC_SMEM 144
// Row pairs per CTA of the rows kernels (RT_ROW_L, /2 or /4) and columns per CTA of the cols kernels (RT_COL_L, /2 or
// /4): the most that fit in shared memory, 0 when none does.
static int rt_row_lines(int W, int w) {
  const int m = ud_any_line_len(W);
  return ud_halving_lines(ud_any_lines(m, rt_rows_fixed_smem(W, m, w) + RT_STATIC_SMEM, W, UD_SMEM_CTA_MAX, RT_ROW_L),
                          RT_ROW_L);
}
static int rt_col_lines(int H) {
  const int m = ud_any_line_len(H);
  return ud_halving_lines(ud_any_lines(m, sizeof(float2) * (size_t)m + RT_STATIC_SMEM, 0, UD_SMEM_CTA_MAX, RT_COL_L),
                          RT_COL_L);
}

static size_t rt_plane_bytes(int H, int W) {
  const size_t v1 = (size_t)H * rt_whp(W) * sizeof(float2), v2 = ud_rt2_workspace_plane_bytes(H, W);
  return v1 > v2 ? v1 : v2;
}

static int rt_chunk_samples(int N, int C, int H, int W) {
  // the Y/T workspace of a chunk must stay L2-resident (126 MB) next to the streamed images
  const size_t per_sample = (size_t)C * rt_plane_bytes(H, W);
  int chunk = (int)((64ull << 20) / (per_sample ? per_sample : 1));
  if (chunk < 1) chunk = 1;
  if (chunk > N) chunk = N;
  return chunk;
}

extern "C" size_t ud_recon_tail_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  (void)h;
  const int chunk = rt_chunk_samples(N, C, H, W);
  // the first-generation tiles outnumber the second generation's; a size no count fits is rejected by the entry points
  const int LR = rt_row_lines(W, w), LC = rt_col_lines(H);
  const int row_tiles = ud_cdiv(H, 2 * (LR > 0 ? LR : 1)), col_tiles = ud_cdiv(W / 2 + 1, LC > 0 ? LC : 1);
  size_t y = ud_align_up((size_t)chunk * C * rt_plane_bytes(H, W), 256);
  size_t ps = ud_align_up((size_t)N * C * row_tiles * sizeof(float), 256);
  size_t pf = ud_align_up((size_t)N * C * col_tiles * sizeof(float), 256);
  return y + ps + pf;
}

extern "C" size_t ud_recon_tail_signs_bytes(int N, int C, int H, int W) {
  return (size_t)N * C * (W / 2 + 1) * H;
}

template <class K>
static int rt_set_smem(K kernel, size_t bytes) {
  if (bytes > (227u << 10)) {
    ud_set_error("recon_tail: needs %zu bytes of shared memory per CTA (> 227 KB)", bytes);
    return UD_ERR_UNSUPPORTED;
  }
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    ud_set_error("cudaFuncSetAttribute(smem=%zu) failed: %s", bytes, cudaGetErrorString(e));
    return UD_ERR_CUDA;
  }
  return UD_OK;
}

static int rt_validate(int N, int C, int h, int w, int H, int W) {
  UD_REQUIRE(N >= 0 && C >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID,
             "recon_tail: bad shape N=%d C=%d h=%d w=%d H=%d W=%d", N, C, h, w, H, W);
  UD_REQUIRE(H <= UD_FFT_MAX_N && W <= UD_FFT_MAX_N, UD_ERR_UNSUPPORTED,
             "recon_tail: FFT size %dx%d unsupported (n <= %d)", H, W, UD_FFT_MAX_N);
  UD_REQUIRE((long long)N * C <= 65535LL * 64, UD_ERR_UNSUPPORTED, "recon_tail: too many planes");
  UD_REQUIRE(rt_row_lines(W, w) > 0, UD_ERR_UNSUPPORTED,
             "recon_tail: %d-point rows with a %d-wide decoder do not fit shared memory", W, w);
  UD_REQUIRE(rt_col_lines(H) > 0, UD_ERR_UNSUPPORTED, "recon_tail: %d-point columns do not fit shared memory", H);
  return UD_OK;
}

extern "C" int ud_recon_tail_fwd(const float* dec, const float* x, float* rec, float* spatial, float* freq,
                                 uint8_t* signs, void* ws, size_t ws_bytes, int N, int C, int h, int w, int H,
                                 int W, int norm_ortho, cudaStream_t stream) {
  int rc = rt_validate(N, C, h, w, H, W);
  if (rc != UD_OK) return rc;
  if (N == 0) return UD_OK;
  UD_REQUIRE(dec && x && rec && spatial && freq && ws, UD_ERR_INVALID, "recon_tail_fwd: null pointer");
  UD_REQUIRE(ws_bytes >= ud_recon_tail_workspace_bytes(N, C, h, w, H, W), UD_ERR_WORKSPACE,
             "recon_tail_fwd: workspace too small (%zu < %zu)", ws_bytes,
             ud_recon_tail_workspace_bytes(N, C, h, w, H, W));
  int chunk = rt_chunk_samples(N, C, H, W);
  if (chunk * C > 65535) chunk = 65535 / C;
  const int Wh = W / 2 + 1;
  const bool v2 = ud_rt2_supported(h, w, H, W);
  const int LR = rt_row_lines(W, w), LC = rt_col_lines(H);
  const int row_tiles = v2 ? ud_cdiv((H + 1) / 2, ud_rt2_rows_lpc()) : ud_cdiv(H, 2 * LR);
  const int col_tiles = v2 ? ud_cdiv(Wh, RT2_COLS_PER_TILE) : ud_cdiv(Wh, LC);
  char* p = static_cast<char*>(ws);
  float2* Y = reinterpret_cast<float2*>(p);
  p += ud_align_up((size_t)rt_chunk_samples(N, C, H, W) * C * rt_plane_bytes(H, W), 256);
  float* part_sp = reinterpret_cast<float*>(p);
  p += ud_align_up((size_t)N * C * row_tiles * sizeof(float), 256);
  float* part_fr = reinterpret_cast<float*>(p);
  UdAnyPlan pW, pH;   // line FFTs of the first-generation kernels: mixed radix, or Bluestein for a prime factor > 23
  if (!ud_make_any_plan(W, &pW) || !ud_make_any_plan(H, &pH)) return UD_ERR_UNSUPPORTED;
  const float2* ytab = ud_lerp_table(h, H);
  const float2* xtab = ud_lerp_table(w, W);
  if (!ytab || !xtab) return UD_ERR_CUDA;
  const size_t smW = rt_rows_smem(W, pW.m, w, LR), smH = rt_cols_smem(pH.m, LC);

  for (int s0 = 0; s0 < N; s0 += chunk) {
    const int ns = (N - s0 < chunk) ? (N - s0) : chunk;
    const int planes = ns * C, plane0 = s0 * C;
    if (v2) {
      if ((rc = ud_rt2_fwd(dec, x, rec, Y, part_sp, part_fr, signs, plane0, planes, h, w, H, W, row_tiles, col_tiles,
                           stream)) != UD_OK) return rc;
      continue;
    }
    UD_LINES_DISPATCH(LR, RT_ROW_L, LV, {
      auto k = rt_rows_fwd_kernel<UdAnyPlan, LV>;
      if ((rc = rt_set_smem(k, smW)) != UD_OK) return rc;
      k<<<dim3(row_tiles, planes), RT_ROW_T, smW, stream>>>(pW, dec, x, rec, Y, part_sp, pW.tw, ytab, xtab, plane0, h, w,
                                                            H, W, row_tiles);
    });
    if ((rc = ud_check_launch("rt_rows_fwd")) != UD_OK) return rc;
    UD_LINES_DISPATCH(LC, RT_COL_L, LV, {
      auto k = rt_cols_fwd_kernel<UdAnyPlan, LV>;
      if ((rc = rt_set_smem(k, smH)) != UD_OK) return rc;
      k<<<dim3(col_tiles, planes), RT_COL_T, smH, stream>>>(pH, Y, part_fr, signs, pH.tw, plane0, H, W, col_tiles);
    });
    if ((rc = ud_check_launch("rt_cols_fwd")) != UD_OK) return rc;
  }
  const float nrm = norm_ortho ? 1.f / sqrtf((float)H * (float)W) : 1.f;
  rt_finalize_kernel<<<N, 128, 0, stream>>>(part_sp, part_fr, spatial, freq, C, row_tiles, col_tiles,
                                            1.f / ((float)C * H * W), nrm / ((float)C * H * Wh));
  return ud_check_launch("rt_finalize");
}

// g_dec and g_x are each nullable (not both); g_x = NULL selects the GX = false kernels (the training path)
extern "C" int ud_recon_tail_bwd(const float* dec, const float* x, const uint8_t* signs, const float* g_spatial,
                                 const float* g_freq, float* g_dec, float* g_x, void* ws, size_t ws_bytes, int N, int C,
                                 int h, int w, int H, int W, int norm_ortho, cudaStream_t stream) {
  int rc = rt_validate(N, C, h, w, H, W);
  if (rc != UD_OK) return rc;
  if (N == 0) return UD_OK;
  UD_REQUIRE(dec && x && signs && g_spatial && g_freq && (g_dec || g_x) && ws, UD_ERR_INVALID,
             "recon_tail_bwd: null pointer");
  UD_REQUIRE(ws_bytes >= ud_recon_tail_workspace_bytes(N, C, h, w, H, W), UD_ERR_WORKSPACE,
             "recon_tail_bwd: workspace too small");
  int chunk = rt_chunk_samples(N, C, H, W);
  if (chunk * C > 65535) chunk = 65535 / C;
  const int Wh = W / 2 + 1;
  const bool v2 = ud_rt2_supported(h, w, H, W);
  const int LR = rt_row_lines(W, w), LC = rt_col_lines(H);
  const int row_tiles = v2 ? ud_cdiv((H + 1) / 2, ud_rt2_rows_lpc()) : ud_cdiv(H, 2 * LR);
  const int col_tiles = v2 ? ud_cdiv(Wh, RT2_COLS_PER_TILE) : ud_cdiv(Wh, LC);
  float2* T = reinterpret_cast<float2*>(ws);
  UdAnyPlan pW, pH;   // line FFTs of the first-generation kernels: mixed radix, or Bluestein for a prime factor > 23
  if (!ud_make_any_plan(W, &pW) || !ud_make_any_plan(H, &pH)) return UD_ERR_UNSUPPORTED;
  const float2* ytab = ud_lerp_table(h, H);
  const float2* xtab = ud_lerp_table(w, W);
  if (!ytab || !xtab) return UD_ERR_CUDA;
  const int2* jtab = ud_lerp_ranges(w, W);
  if (!jtab) return UD_ERR_CUDA;
  const size_t smH = rt_cols_smem(pH.m, LC), smW = rt_rows_smem(W, pW.m, w, LR);
  // freq[n] = nrm/(C*H*Wh) * sum |D'| with D' the unnormalised spectrum, so the sign spectrum
  // carries nrm/(C*H*Wh) and the adjoint of the unnormalised forward is the unnormalised inverse.
  const float nrm = norm_ortho ? 1.f / sqrtf((float)H * (float)W) : 1.f;
  const float gscale = nrm / ((float)C * H * Wh);
  const float sp_scale = 1.f / ((float)C * H * W);
  if (g_dec) UD_CUDA(cudaMemsetAsync(g_dec, 0, sizeof(float) * (size_t)N * C * h * w, stream));
  for (int s0 = 0; s0 < N; s0 += chunk) {
    const int ns = (N - s0 < chunk) ? (N - s0) : chunk;
    const int planes = ns * C, plane0 = s0 * C;
    if (v2) {
      if ((rc = ud_rt2_bwd(dec, x, signs, g_spatial, g_freq, g_dec, g_x, T, plane0, planes, C, h, w, H, W, row_tiles, col_tiles,
                           gscale, sp_scale, stream)) != UD_OK) return rc;
      continue;
    }
    UD_LINES_DISPATCH(LC, RT_COL_L, LV, {
      auto k = rt_cols_bwd_kernel<UdAnyPlan, LV>;
      if ((rc = rt_set_smem(k, smH)) != UD_OK) return rc;
      k<<<dim3(col_tiles, planes), RT_COL_T, smH, stream>>>(pH, signs, g_freq, T, pH.tw, plane0, C, H, W, gscale);
    });
    if ((rc = ud_check_launch("rt_cols_bwd")) != UD_OK) return rc;
    UD_LINES_DISPATCH(LR, RT_ROW_L, LV, {
      auto k = g_x ? rt_rows_bwd_kernel<UdAnyPlan, true, LV> : rt_rows_bwd_kernel<UdAnyPlan, false, LV>;
      if ((rc = rt_set_smem(k, smW)) != UD_OK) return rc;
      k<<<dim3(row_tiles, planes), RT_ROW_T, smW, stream>>>(pW, dec, x, T, g_spatial, g_freq, g_dec, g_x, pW.tw, ytab,
                                                             xtab, jtab, plane0, C, h, w, H, W, sp_scale);
    });
    if ((rc = ud_check_launch("rt_rows_bwd")) != UD_OK) return rc;
  }
  return UD_OK;
}
