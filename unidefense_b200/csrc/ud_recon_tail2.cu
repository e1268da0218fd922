// a1 -- reconstruction-loss tail, second-generation kernels for the configured image sizes
//                                                                     (SURVEY.md §8a row a1)
// Same math, entry points and saved state as ud_recon_tail.cu (reference: model/unidefense.py:244-253, :423-433,
// :618-628; backward = torch autograd of those lines), rebuilt around the register-resident two-stage line FFT of
// ud_fft.cuh (Ud2S) for the configured lengths (UdConfigured):
//   * a line (two packed image rows, or one spectrum column) is owned by 20 (16, 23) threads whose roles never
//     change, so the butterflies carry no index arithmetic and the pixel work happens in the registers the
//     radix-R1 butterfly consumes: x is read and rec written straight from/to global memory, 4 bytes per lane,
//     R2 consecutive floats per line and instruction;
//   * ONE shared-memory exchange and ONE barrier per line instead of one (two, in place) per radix stage;
//   * the row pass stores the PACKED row spectra Z[pair][k] (two real rows per complex line); the unpack
//     A[k] = (Z[k] + conj Z[n-k])/2, B[k] = (Z[k] - conj Z[n-k])/2i happens while the column pass loads its
//     columns k and n-k -- no cross-thread unpack, and the workspace is the same size as before;
//   * backward: inverse column FFTs straight from the sign bytes, Hermitian fold + packed inverse row FFT from
//     registers, sign(rec - x) recomputed in place, transposed bilinear resize as a horizontal gather plus a
//     per-column walk that keeps its running sums in registers across the whole tile (one atomicAdd per finished
//     decoder row).
// Sizes without a two-factor plan keep using the shared-memory Stockham kernels of ud_recon_tail.cu.
#include "../../include/unidefense_b200.h"
#include "ud_fft.cuh"

#define RT2_LPC 16    // columns per CTA step of the cols kernels (16 float2 = one 128-byte line per row)
#ifndef RT2_RLPC
// row pairs per CTA step of the rows kernels (threads = TL * RT2_RLPC).  Measured at N=32, 380^2 (fwd / bwd us): 16 ->
// 101 / 89 (96 registers, 376 B spilled in rows_bwd, 20 warps per SM); 12 -> 110 / 95 and 10 -> 112 / 105 (128 registers,
// fewer spills, 15 warps per SM): resident warps matter more than the spills.
#define RT2_RLPC 16
#endif
// row-pair steps per CTA of the rows kernels: a launch parameter (`iters`, derived from the row-tile count the caller chose)

// Vertical lerps of the row pair of line g (vertical first, like ud_recon_tail.cu): V[c] = (row 2p, row 2p+1) of the
// upsampled image BEFORE the horizontal lerp.  The TL threads of the line stride over the dec columns; the row taps
// are decoded once per thread and the four row pointers hoisted, so an item costs 4 coalesced loads + 4 flops.
template <int TL>
__device__ __forceinline__ void rt2_vrows(const float* __restrict__ decp, const float2* __restrict__ ytab_g, int ra, int ln,
                                          int h, int w, int H, float2* __restrict__ Vg) {
  if (ra >= H) {
    for (int c = ln; c < w; c += TL) Vg[c] = make_float2(0.f, 0.f);
    return;
  }
  int a0, a1, b0, b1;
  float la0, la1, lb0, lb1;
  ud_lerp_tab(__ldg(ytab_g + ra), h, a0, a1, la0, la1);
  const bool has_b = ra + 1 < H;
  ud_lerp_tab(__ldg(ytab_g + (has_b ? ra + 1 : ra)), h, b0, b1, lb0, lb1);
  if (!has_b) lb0 = lb1 = 0.f;
  const float* pa0 = decp + (long long)a0 * w;
  const float* pa1 = decp + (long long)a1 * w;
  const float* pb0 = decp + (long long)b0 * w;
  const float* pb1 = decp + (long long)b1 * w;
#pragma unroll 4
  for (int c = ln; c < w; c += TL)
    Vg[c] = make_float2(la0 * __ldg(pa0 + c) + la1 * __ldg(pa1 + c), lb0 * __ldg(pb0 + c) + lb1 * __ldg(pb1 + c));
}

// ------------------------------------------------------------------------------------------
// forward rows: grid (row_tiles, planes_in_chunk), PL::TL * RT2_RLPC threads
//   shared: tw2[R1*P] | xtab[N] | S[LPC*LS] | V[LPC*w]
// ------------------------------------------------------------------------------------------
template <class PL>
__global__ void __launch_bounds__(PL::TL* RT2_RLPC, 2)
rt2_rows_fwd_kernel(const float* __restrict__ dec, const float* __restrict__ x, float* __restrict__ rec,
                    float2* __restrict__ Z, float* __restrict__ part_spatial, const float2* __restrict__ tw_g,
                    const float2* __restrict__ ytab_g, const float2* __restrict__ xtab_g, int plane0, int h, int w, int H,
                    int row_tiles, int iters) {
  constexpr int N = PL::N, R1 = PL::R1, R2 = PL::R2, TL = PL::TL, P = PL::P, LS = PL::LS;
  extern __shared__ float2 smem[];
  float2* tw2 = smem;
  float2* xtab = tw2 + R1 * P;
  float2* S = xtab + N;
  float2* V = S + RT2_RLPC * LS;
  __shared__ float red[33];
  const int tid = threadIdx.x, g = tid / TL, ln = tid - g * TL;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int Hp = (H + 1) >> 1;
  const int pair0 = blockIdx.x * (RT2_RLPC * iters);

  ud2s_build_tw<PL>(tw2, tw_g);
  for (int t = tid; t < N; t += TL * RT2_RLPC) xtab[t] = __ldg(xtab_g + t);
  const float* decp = dec + plane * (long long)h * w;
  const float* xp = x + plane * (long long)H * N;
  float* recp = rec + plane * (long long)H * N;
  float2* Zp = Z + (long long)pl * Hp * N;
  float acc = 0.f;
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
    const int pbase = pair0 + it * RT2_RLPC;
    if (pbase >= Hp) break;
    const int p = pbase + g, ra = 2 * p;
    const bool live = ra < H, has_b = ra + 1 < H;
    rt2_vrows<TL>(decp, ytab_g, ra, ln, h, w, H, V + g * w);
    __syncthreads();       // V (and, first time, tw2/xtab) visible; everyone is past the previous step's S reads
    if (live && ln < R2) {
      float2 z[R1];
      const float* xa = xp + (long long)ra * N;
      float* qa = recp + (long long)ra * N;
      const float2* Vg = V + g * w;
#pragma unroll
      for (int n1 = 0; n1 < R1; ++n1) {
        const int c = ln + R2 * n1;
        int i0, i1;
        float l0, l1;
        ud_lerp_tab(xtab[c], w, i0, i1, l0, l1);
        const float2 v0 = Vg[i0], v1 = Vg[i1];
        const float va = l0 * v0.x + l1 * v1.x;
        __stcs(qa + c, va);
        const float dA = va - __ldcs(xa + c);
        float dB = 0.f;
        if (has_b) {
          const float vb = l0 * v0.y + l1 * v1.y;
          __stcs(qa + N + c, vb);
          dB = vb - __ldcs(xa + N + c);
        }
        acc += fabsf(dA) + fabsf(dB);
        z[n1] = make_float2(dA, dB);
      }
      ud2s_stage_a<PL>(z, ln, tw2, S + g * LS);
    }
    __syncthreads();
    if (live && ln < R1) {
      float2 u[R2];
      ud2s_stage_b<PL>(u, ln, S + g * LS);
      float2* zr = Zp + (long long)p * N;
#pragma unroll
      for (int k2 = 0; k2 < R2; ++k2) zr[ln + R1 * k2] = u[k2];
    }
  }
  const float tot = ud_block_sum(acc, red);
  if (tid == 0) part_spatial[plane * row_tiles + blockIdx.x] = tot;
}

// ------------------------------------------------------------------------------------------
// forward cols: PERSISTENT, grid = min(tiles, 2 * SMs); a tile = 16 spectrum columns of one plane.  PL is the plan
// of the column length H; Wn = row length.  While a tile is transformed, the packed row spectra of the NEXT tile
// (columns k and Wn-k, 128-byte row segments) are already in flight into the other stage buffer (cp.async), so
// the L2/HBM latency of the load phase is hidden behind the butterflies.  The unpack of the two real rows of a
// pair happens when stage A gathers its registers.
//   shared: tw2[R1*P] | stage[2][LPC*SB], SB = max(2*HPP, LS): per line K part [p], M part [HPP + p]; the
//   exchange buffer of stage A/B aliases the stage that has just been consumed.
// ------------------------------------------------------------------------------------------
template <class PL>
struct Rt2Cols {
  static constexpr int Hp = (PL::N + 1) / 2;
  static constexpr int HPP = Hp | 1;
  static constexpr int SB = (2 * HPP > PL::LS ? 2 * HPP : PL::LS) | 1;
};

template <class PL>
__device__ __forceinline__ void rt2_cols_issue(const float2* __restrict__ Z, float2* __restrict__ st, int tile, int col_tiles,
                                               int Wn) {
  constexpr int Hp = Rt2Cols<PL>::Hp, HPP = Rt2Cols<PL>::HPP, SB = Rt2Cols<PL>::SB;
  const int pl = tile / col_tiles, ct = tile - pl * col_tiles;
  const int Wh = Wn / 2 + 1;
  const int k0 = ct * RT2_LPC;
  const int ncols = min(RT2_LPC, Wh - k0);
  const float2* Zp = Z + (long long)pl * Hp * Wn;
  for (int idx = threadIdx.x; idx < Hp * RT2_LPC; idx += PL::TL * RT2_LPC) {
    const int p = idx / RT2_LPC, j = idx - p * RT2_LPC;
    float2* d = st + j * SB + p;
    if (j < ncols) {
      const int k = k0 + j;
      ud_cp_async8(d, Zp + (long long)p * Wn + k);
      ud_cp_async8(d + HPP, Zp + (long long)p * Wn + (k == 0 ? 0 : Wn - k));
    } else {
      d[0] = make_float2(0.f, 0.f);
      d[HPP] = make_float2(0.f, 0.f);
    }
  }
}

template <class PL>
__global__ void __launch_bounds__(PL::TL* RT2_LPC, 2)
rt2_cols_fwd_kernel(const float2* __restrict__ Z, float* __restrict__ part_freq, uint8_t* __restrict__ signs,
                    const float2* __restrict__ tw_g, int plane0, int planes, int Wn, int col_tiles) {
  constexpr int H = PL::N, R1 = PL::R1, R2 = PL::R2, TL = PL::TL, P = PL::P;
  constexpr int HPP = Rt2Cols<PL>::HPP, SB = Rt2Cols<PL>::SB;
  extern __shared__ float2 smem[];
  float2* tw2 = smem;
  float2* stage0 = tw2 + R1 * P;
  __shared__ float red[33];
  const int tid = threadIdx.x, g = tid / TL, ln = tid - g * TL;
  const int Wh = Wn / 2 + 1;
  const int total = planes * col_tiles;
  ud2s_build_tw<PL>(tw2, tw_g);
  int tile = blockIdx.x;
  if (tile < total) rt2_cols_issue<PL>(Z, stage0, tile, col_tiles, Wn);
  ud_cp_async_commit();
  int sidx = 0;
#pragma unroll 1
  for (; tile < total; tile += gridDim.x, sidx ^= 1) {
    float2* st = stage0 + sidx * (RT2_LPC * SB);
    const int nxt = tile + gridDim.x;
    if (nxt < total) rt2_cols_issue<PL>(Z, stage0 + (sidx ^ 1) * (RT2_LPC * SB), nxt, col_tiles, Wn);
    ud_cp_async_commit();
    asm volatile("cp.async.wait_group 1;\n" ::: "memory");      // this tile's loads have landed (the next may fly)
    __syncthreads();
    const int pl = tile / col_tiles, ct = tile - pl * col_tiles;
    const long long plane = plane0 + pl;
    const int k0 = ct * RT2_LPC;
    const int ncols = min(RT2_LPC, Wh - k0);
    float2 z[R1];
    if (ln < R2) {
      const float2* sk = st + g * SB;
#pragma unroll
      for (int n1 = 0; n1 < R1; ++n1) {
        const int r = ln + R2 * n1;
        const float2 z1 = sk[r >> 1], z2 = sk[HPP + (r >> 1)];
        // row 2p: (Z[k] + conj Z[n-k]) / 2 ; row 2p+1: (Z[k] - conj Z[n-k]) / 2i
        z[n1] = (r & 1) ? make_float2(0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x))
                        : make_float2(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y));
      }
    }
    __syncthreads();
    if (ln < R2) ud2s_stage_a<PL>(z, ln, tw2, st + g * SB);
    __syncthreads();
    float acc = 0.f;
    if (ln < R1) {
      float2 u[R2];
      ud2s_stage_b<PL>(u, ln, st + g * SB);
      const bool wr = signs != nullptr && g < ncols;
      uint8_t* sg = signs + (plane * Wh + (k0 + g)) * (long long)H;
#pragma unroll
      for (int k2 = 0; k2 < R2; ++k2) {
        const float2 v = u[k2];
        acc += fabsf(v.x) + fabsf(v.y);
        if (wr) {
          const uint8_t sr = v.x > 0.f ? 1 : (v.x < 0.f ? 2 : 0);
          const uint8_t si = v.y > 0.f ? 1 : (v.y < 0.f ? 2 : 0);
          sg[ln + R1 * k2] = (uint8_t)(sr | (si << 2));
        }
      }
    }
    const float tot = ud_block_sum(acc, red);      // its barriers also fence the stage buffer for the next issue
    if (tid == 0) part_freq[plane * col_tiles + ct] = tot;
  }
  asm volatile("cp.async.wait_all;\n" ::: "memory");
}

// ------------------------------------------------------------------------------------------
// backward cols: inverse column FFT of the sign spectrum (swap trick), T[r][k] written as 128-byte row segments
//   shared: tw2[R1*P] | buf[max(LPC*LS, H*(LPC+1))]
// ------------------------------------------------------------------------------------------
template <class PL>
__global__ void __launch_bounds__(PL::TL* RT2_LPC, 2)
rt2_cols_bwd_kernel(const uint8_t* __restrict__ signs, const float* __restrict__ g_freq, float2* __restrict__ T,
                    const float2* __restrict__ tw_g, int plane0, int C, int Wn, float gscale) {
  constexpr int H = PL::N, R1 = PL::R1, R2 = PL::R2, TL = PL::TL, P = PL::P, LS = PL::LS;
  extern __shared__ float2 smem[];
  float2* tw2 = smem;
  float2* buf = tw2 + R1 * P;
  const int tid = threadIdx.x, g = tid / TL, ln = tid - g * TL;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int smp = (int)(plane / C);
  const float gfs = __ldg(g_freq + smp);
  if (gfs == 0.f) return;                 // the rows kernel skips the FFT of this plane too
  const float gf = gfs * gscale;
  const int Wh = Wn / 2 + 1;
  const int WhP = (Wh + 15) & ~15;
  const int k0 = blockIdx.x * RT2_LPC;
  const int ncols = min(RT2_LPC, Wh - k0);
  ud2s_build_tw<PL>(tw2, tw_g);
  __syncthreads();
  if (ln < R2) {
    float2 z[R1];
    const uint8_t* sg = signs + (plane * Wh + (k0 + g)) * (long long)H;
#pragma unroll
    for (int n1 = 0; n1 < R1; ++n1) {
      float2 v = make_float2(0.f, 0.f);
      if (g < ncols) {
        const uint8_t s = __ldg(sg + ln + R2 * n1);
        const float sr = (s & 1) ? gf : ((s & 2) ? -gf : 0.f);
        const float si = (s & 4) ? gf : ((s & 8) ? -gf : 0.f);
        v = make_float2(si, sr);          // swapped: IFFT(z) = swap(FFT(swap(z)))
      }
      z[n1] = v;
    }
    ud2s_stage_a<PL>(z, ln, tw2, buf + g * LS);
  }
  __syncthreads();
  float2 u[R2];
  if (ln < R1) ud2s_stage_b<PL>(u, ln, buf + g * LS);
  __syncthreads();                        // every line's exchange buffer has been read: reuse buf as out[H][LPC+1]
  if (ln < R1) {
#pragma unroll
    for (int k2 = 0; k2 < R2; ++k2) buf[(ln + R1 * k2) * (RT2_LPC + 1) + g] = make_float2(u[k2].y, u[k2].x);
  }
  __syncthreads();
  float2* Tp = T + (long long)pl * H * WhP;
  for (int idx = tid; idx < H * RT2_LPC; idx += TL * RT2_LPC) {
    const int r = idx / RT2_LPC, j = idx - r * RT2_LPC;
    if (j < ncols) Tp[(long long)r * WhP + k0 + j] = buf[r * (RT2_LPC + 1) + j];
  }
}

// ------------------------------------------------------------------------------------------
// backward rows: grid (row_tiles, planes_in_chunk)
//   g_rec[r,c] = gs*sign(d[r,c]) + Re sum_{k<Wh} T[r,k] e^{+2 pi i k c / W}; transposed bilinear into g_dec.
//   GX: also g_x = -g_rec at full resolution, straight from the registers that hold g_rec (zeros for planes whose
//   sample has gs == gf == 0); g_dec may then be NULL (no transposed resize).  GX = false is the training path.
//   shared: tw2[R1*P] | xtab[N] | S[LPC*LS] | V[LPC*w] (aliased by Hb[2*LPC][w] floats)
// ------------------------------------------------------------------------------------------
template <class PL, bool GX>
__global__ void __launch_bounds__(PL::TL* RT2_RLPC, 2)
rt2_rows_bwd_kernel(const float* __restrict__ dec, const float* __restrict__ x, const float2* __restrict__ T,
                    const float* __restrict__ g_spatial, const float* __restrict__ g_freq, float* __restrict__ g_dec,
                    float* __restrict__ g_x, const float2* __restrict__ tw_g, const float2* __restrict__ ytab_g,
                    const float2* __restrict__ xtab_g, const int2* __restrict__ jtab_g, int plane0, int C, int h, int w,
                    int H, float sp_scale, int iters) {
  constexpr int N = PL::N, R1 = PL::R1, R2 = PL::R2, TL = PL::TL, P = PL::P, LS = PL::LS;
  constexpr int NT = TL * RT2_RLPC;
  extern __shared__ float2 smem[];
  float2* tw2 = smem;
  float2* xtab = tw2 + R1 * P;
  float2* S = xtab + N;
  float2* V = S + RT2_RLPC * LS;
  float* Hb = reinterpret_cast<float*>(V);            // [2*LPC][w] floats == LPC*w float2
  const int tid = threadIdx.x, g = tid / TL, ln = tid - g * TL;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int smp = (int)(plane / C);
  const float gs = __ldg(g_spatial + smp) * sp_scale;
  const bool has_f = __ldg(g_freq + smp) != 0.f;
  const int Hp = (H + 1) >> 1;
  const int pair0 = blockIdx.x * (RT2_RLPC * iters);
  if (gs == 0.f && !has_f) {
    if (GX) {                              // the tile's rows of g_x are zero
      const int r0 = 2 * pair0, r1 = min(H, 2 * (pair0 + RT2_RLPC * iters));
      float* gxp = g_x + plane * (long long)H * N;
      for (long long i = (long long)r0 * N + tid; i < (long long)r1 * N; i += NT) gxp[i] = 0.f;
    }
    return;
  }
  const int Wh = N / 2 + 1;
  const int WhP = (Wh + 15) & ~15;

  ud2s_build_tw<PL>(tw2, tw_g);
  for (int t = tid; t < N; t += NT) xtab[t] = __ldg(xtab_g + t);
  const float* decp = dec + plane * (long long)h * w;
  const float* xp = x + plane * (long long)H * N;
  const float2* Tp = T + (long long)pl * H * WhP;
  float* gd = g_dec + plane * (long long)h * w;
  // vertical walk state of dec column `tid` (threads < w), carried across the steps of the tile
  int cur = 0;
  float acc0 = 0.f, acc1 = 0.f;
  if (tid < w && 2 * pair0 < H) cur = __float_as_int(__ldg(ytab_g + 2 * pair0).x);
#pragma unroll 1
  for (int it = 0; it < iters; ++it) {
    const int pbase = pair0 + it * RT2_RLPC;
    if (pbase >= Hp) break;
    const int p = pbase + g, ra = 2 * p;
    const bool live = ra < H, has_b = ra + 1 < H;
    if (gs != 0.f) rt2_vrows<TL>(decp, ytab_g, ra, ln, h, w, H, V + g * w);
    if (has_f && live && ln < R2) {
      // V[k] = Th_a[k] + i Th_b[k], Th = Hermitian fold of the zero-padded half spectrum; stored swapped
      float2 z[R1];
      const float2* ta_p = Tp + (long long)ra * WhP;
#pragma unroll
      for (int n1 = 0; n1 < R1; ++n1) {
        const int k = ln + R2 * n1;
        const int kk = (k < Wh) ? k : N - k;
        const float2 ta = __ldg(ta_p + kk);
        const float2 tb = has_b ? __ldg(ta_p + WhP + kk) : make_float2(0.f, 0.f);
        float2 v;
        if (k == 0 || 2 * k == N) {
          v = make_float2(tb.x, ta.x);
        } else {
          const float ar = 0.5f * ta.x, ai = 0.5f * ta.y, br = 0.5f * tb.x, bi = 0.5f * tb.y;
          v = (k < Wh) ? make_float2(ai + br, ar - bi) : make_float2(br - ai, ar + bi);
        }
        z[n1] = v;
      }
      ud2s_stage_a<PL>(z, ln, tw2, S + g * LS);
    }
    __syncthreads();                       // S and V ready
    float2 u[R2];
    if (live && ln < R1) {
      if (has_f) {
        ud2s_stage_b<PL>(u, ln, S + g * LS);       // u[k2] = (g_b[c], g_a[c]), c = ln + R1*k2
      } else {
#pragma unroll
        for (int k2 = 0; k2 < R2; ++k2) u[k2] = make_float2(0.f, 0.f);
      }
      if (gs != 0.f) {                     // + gs * sign(rec - x)
        const float* xa = xp + (long long)ra * N;
        const float2* Vg = V + g * w;
#pragma unroll
        for (int k2 = 0; k2 < R2; ++k2) {
          const int c = ln + R1 * k2;
          int i0, i1;
          float l0, l1;
          ud_lerp_tab(xtab[c], w, i0, i1, l0, l1);
          const float2 v0 = Vg[i0], v1 = Vg[i1];
          const float dA = (l0 * v0.x + l1 * v1.x) - __ldcs(xa + c);
          u[k2].y += dA > 0.f ? gs : (dA < 0.f ? -gs : 0.f);
          if (has_b) {
            const float dB = (l0 * v0.y + l1 * v1.y) - __ldcs(xa + N + c);
            u[k2].x += dB > 0.f ? gs : (dB < 0.f ? -gs : 0.f);
          }
        }
      }
    }
    if (GX && live && ln < R1) {           // g_x = -g_rec: u[k2] = (g_b[c], g_a[c])
      float* qa = g_x + (plane * H + ra) * (long long)N;
#pragma unroll
      for (int k2 = 0; k2 < R2; ++k2) {
        const int c = ln + R1 * k2;
        __stcs(qa + c, -u[k2].y);
        if (has_b) __stcs(qa + N + c, -u[k2].x);
      }
    }
    __syncthreads();                       // all reads of S (stage B) and V (signs) done
    if (GX && g_dec == nullptr) continue;  // g_x only: no transposed resize
    if (ln < R1) {
      float2* Gg = S + g * LS;             // G[c] = (g_b[c], g_a[c]); dead lines hold zeros
#pragma unroll
      for (int k2 = 0; k2 < R2; ++k2) Gg[ln + R1 * k2] = live ? u[k2] : make_float2(0.f, 0.f);
    }
    __syncthreads();
    // horizontal transposed lerp: Hb[2*gg + {0,1}][j] for every dec column j of every line
    for (int idx = tid; idx < RT2_RLPC * w; idx += NT) {
      const int gg = idx / w, j = idx - gg * w;
      const int2 cr = __ldg(jtab_g + j);
      const float2* Gg = S + gg * LS;
      float ax = 0.f, ay = 0.f;
      for (int c = cr.x; c <= cr.y; ++c) {
        const float2 t = xtab[c];
        const int i0 = __float_as_int(t.x);
        const float wgt = (i0 == j) ? (1.f - t.y) + ((i0 == w - 1) ? t.y : 0.f) : t.y;   // i0 == j-1 -> the l1 tap
        const float2 gv = Gg[c];
        ax = fmaf(wgt, gv.x, ax);
        ay = fmaf(wgt, gv.y, ay);
      }
      Hb[(2 * gg) * w + j] = ay;           // row 2p   (g_a)
      Hb[(2 * gg + 1) * w + j] = ax;       // row 2p+1 (g_b)
    }
    __syncthreads();
    // vertical transposed lerp: thread j walks the rows of this step in order, two running sums
    if (tid < w) {
      const int r0 = 2 * pbase;
      const int nrows = min(2 * RT2_RLPC, H - r0);
      for (int rr = 0; rr < nrows; ++rr) {
        int i0, i1;
        float l0, l1;
        ud_lerp_tab(__ldg(ytab_g + r0 + rr), h, i0, i1, l0, l1);
        while (cur < i0) {
          if (acc0 != 0.f) atomicAdd(gd + (long long)cur * w + tid, acc0);
          acc0 = acc1;
          acc1 = 0.f;
          ++cur;
        }
        const float v = Hb[rr * w + tid];
        acc0 = fmaf(l0, v, acc0);
        if (i1 > i0) acc1 = fmaf(l1, v, acc1);
        else acc0 = fmaf(l1, v, acc0);
      }
    }
    __syncthreads();                       // Hb (== V) and S are rewritten by the next step
  }
  if (GX && g_dec == nullptr) return;
  if (tid < w) {
    if (acc0 != 0.f) atomicAdd(gd + (long long)cur * w + tid, acc0);
    if (acc1 != 0.f && cur + 1 < h) atomicAdd(gd + (long long)(cur + 1) * w + tid, acc1);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// steps of RT2_RLPC row pairs a rows CTA walks so that `row_tiles` CTAs cover the (H+1)/2 pairs of a plane
int ud_rt2_rows_lpc(void) { return RT2_RLPC; }
static int rt2_iters(int H, int row_tiles) { return ud_cdiv(ud_cdiv((H + 1) / 2, RT2_RLPC), row_tiles); }

// configured lengths only (ud_rt2_fwd / ud_rt2_bwd run only shapes accepted here), and decoder planes at most as wide as
// the widest thread block (the vertical walk uses one thread per dec column)
bool ud_rt2_supported(int h, int w, int H, int W) {
  (void)h;
  if (!ud_fft_configured(H)) return false;
  int tl = 0;
  UD_FFT_CONFIGURED(W, CFG, , tl = CFG::TwoStage::TL);
  return w <= tl * RT2_RLPC && w >= 1;
}

size_t ud_rt2_workspace_plane_bytes(int H, int W) {
  const size_t z = (size_t)((H + 1) / 2) * W * sizeof(float2);                    // packed row spectra (forward)
  const size_t t = (size_t)H * (((W / 2 + 1) + 15) & ~15) * sizeof(float2);       // T (backward)
  return z > t ? z : t;
}

int ud_rt2_fwd(const float* dec, const float* x, float* rec, float2* Z, float* part_sp, float* part_fr, uint8_t* signs,
               int plane0, int planes, int h, int w, int H, int W, int row_tiles, int col_tiles, cudaStream_t stream) {
  const float2* twW = ud_twiddles(W);
  const float2* twH = ud_twiddles(H);
  const float2* ytab = ud_lerp_table(h, H);
  const float2* xtab = ud_lerp_table(w, W);
  if (!twW || !twH || !ytab || !xtab) return UD_ERR_CUDA;
  int rc;
  UD_FFT_CONFIGURED(W, CFG, return UD_ERR_UNSUPPORTED, {
    using PLW = CFG::TwoStage;
    auto k = rt2_rows_fwd_kernel<PLW>;
    const size_t sm = sizeof(float2) * ((size_t)PLW::R1 * PLW::P + W + (size_t)RT2_RLPC * PLW::LS + (size_t)RT2_RLPC * w);
    if ((rc = ud_set_smem(k, sm, "recon_tail")) != UD_OK) return rc;
    k<<<dim3(row_tiles, planes), PLW::TL * RT2_RLPC, sm, stream>>>(dec, x, rec, Z, part_sp, twW, ytab, xtab, plane0, h, w, H,
                                                                    row_tiles, rt2_iters(H, row_tiles));
  });
  if ((rc = ud_check_launch("rt2_rows_fwd")) != UD_OK) return rc;
  UD_FFT_CONFIGURED(H, CFG, return UD_ERR_UNSUPPORTED, {
    using PLH = CFG::TwoStage;
    auto k = rt2_cols_fwd_kernel<PLH>;
    const size_t sm = sizeof(float2) * ((size_t)PLH::R1 * PLH::P + 2ull * RT2_LPC * Rt2Cols<PLH>::SB);
    if ((rc = ud_set_smem(k, sm, "recon_tail")) != UD_OK) return rc;
    const int total = planes * col_tiles;
    const int grid = total < 2 * UD_NUM_SMS ? total : 2 * UD_NUM_SMS;
    k<<<grid, PLH::TL * RT2_LPC, sm, stream>>>(Z, part_fr, signs, twH, plane0, planes, W, col_tiles);
  });
  return ud_check_launch("rt2_cols_fwd");
}

int ud_rt2_bwd(const float* dec, const float* x, const uint8_t* signs, const float* g_spatial, const float* g_freq,
               float* g_dec, float* g_x, float2* T, int plane0, int planes, int C, int h, int w, int H, int W, int row_tiles,
               int col_tiles, float gscale, float sp_scale, cudaStream_t stream) {
  const float2* twW = ud_twiddles(W);
  const float2* twH = ud_twiddles(H);
  const float2* ytab = ud_lerp_table(h, H);
  const float2* xtab = ud_lerp_table(w, W);
  const int2* jtab = ud_lerp_ranges(w, W);
  if (!twW || !twH || !ytab || !xtab || !jtab) return UD_ERR_CUDA;
  int rc;
  UD_FFT_CONFIGURED(H, CFG, return UD_ERR_UNSUPPORTED, {
    using PLH = CFG::TwoStage;
    auto k = rt2_cols_bwd_kernel<PLH>;
    const size_t a = (size_t)RT2_LPC * PLH::LS, b = (size_t)H * (RT2_LPC + 1);
    const size_t sm = sizeof(float2) * ((size_t)PLH::R1 * PLH::P + (a > b ? a : b));
    if ((rc = ud_set_smem(k, sm, "recon_tail")) != UD_OK) return rc;
    k<<<dim3(col_tiles, planes), PLH::TL * RT2_LPC, sm, stream>>>(signs, g_freq, T, twH, plane0, C, W, gscale);
  });
  if ((rc = ud_check_launch("rt2_cols_bwd")) != UD_OK) return rc;
  UD_FFT_CONFIGURED(W, CFG, return UD_ERR_UNSUPPORTED, {
    using PLW = CFG::TwoStage;
    auto k = g_x ? rt2_rows_bwd_kernel<PLW, true> : rt2_rows_bwd_kernel<PLW, false>;
    const size_t sm = sizeof(float2) * ((size_t)PLW::R1 * PLW::P + W + (size_t)RT2_RLPC * PLW::LS + (size_t)RT2_RLPC * w);
    if ((rc = ud_set_smem(k, sm, "recon_tail")) != UD_OK) return rc;
    k<<<dim3(row_tiles, planes), PLW::TL * RT2_RLPC, sm, stream>>>(dec, x, T, g_spatial, g_freq, g_dec, g_x, twW, ytab,
                                                                    xtab, jtab, plane0, C, h, w, H, sp_scale,
                                                                    rt2_iters(H, row_tiles));
  });
  return ud_check_launch("rt2_rows_bwd");
}
