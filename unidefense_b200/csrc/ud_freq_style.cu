// a13 -- FrequencyStyleTransfer: amplitude mix with the content phase (no grad)     (SURVEY.md §8a row a13)
//
// Reference: model/modules.py:35-55
//     Fa = rfft2(content, ortho); Fb = rfft2(style, ortho)
//     out = irfft2((lmda*|Fa| + (1-lmda)*|Fb|) * exp(1j*angle(Fa)), s=(H,W), ortho)       lmda [B] in [0.5,1)
// Three kernels per chunk of samples, spectra never leave the L2-resident workspace:
//   rows : content row r and style row r packed as ONE complex line -> row FFT -> unpack A_r[k], B_r[k]
//   cols : 8 column pairs per CTA: forward column FFTs of A and B, the amplitude/phase mix on the bins,
//          inverse column FFT of the mixed spectrum in the same shared-memory buffer
//   rows^-1 : Hermitian extension (c2r semantics: imaginary parts of the DC / Nyquist columns are ignored),
//          two output rows per complex line, inverse row FFT, 1/(H*W) scaling, coalesced stores.
#include "../../include/unidefense_b200.h"
#include <type_traits>

#include "ud_fft_any.cuh"

#define FS_ROW_T 256
#define FS_ROW_L 12
#define FS_COL_T 320
#define FS_COL_L 16   // lines per cols CTA: 8 content columns + 8 style columns
#define FS_COL_K 8
// Lines longer than shared memory holds at those counts (long Bluestein lines, m = 1024 or 2048) run instantiations
// with a half or a quarter of them: fs_row_lines / fs_col_k pick the largest that fits.

static inline int fs_whp(int W) { return ((W / 2 + 1) + 7) & ~7; }

template <class Plan, int L>
__global__ void __launch_bounds__(FS_ROW_T)
fs_rows_fwd_kernel(Plan plan, const float* __restrict__ a, const float* __restrict__ b, float2* __restrict__ Ya,
                   float2* __restrict__ Yb, const float2* __restrict__ tw_g, int plane0, int H, int W) {
  extern __shared__ float2 smem[];
  const int n = plan.n();
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* buf0 = tw + m;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;
  W = n;
  const int Wh = n / 2 + 1;
  const int WhP = (Wh + 7) & ~7;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int r0 = blockIdx.x * L;
  for (int t = threadIdx.x; t < m; t += FS_ROW_T) tw[t] = __ldg(tw_g + t);
  const float* ap = a + plane * (long long)H * W;
  const float* bp = b + plane * (long long)H * W;
  for (int p = 0; p < L; ++p) {
    const int r = r0 + p;
    float2* line = buf0 + p * LS;
    if (r < H) {
      for (int c = threadIdx.x; c < W; c += FS_ROW_T) {
        ud_cp_async4(&line[c].x, ap + (long long)r * W + c);
        ud_cp_async4(&line[c].y, bp + (long long)r * W + c);
      }
    } else {
      for (int c = threadIdx.x; c < W; c += FS_ROW_T) line[c] = make_float2(0.f, 0.f);
    }
  }
  ud_cp_async_commit();
  ud_cp_async_wait_all();
  __syncthreads();
  float2* res = plan.run(buf0, buf1, tw, L, LS);
  float2* Yap = Ya + (long long)pl * H * WhP;
  float2* Ybp = Yb + (long long)pl * H * WhP;
  for (int t = threadIdx.x; t < L * Wh; t += FS_ROW_T) {
    const int p = t / Wh, k = t - p * Wh;
    const int r = r0 + p;
    if (r >= H) continue;
    const float2 z = res[p * LS + k];
    const float2 zn = res[p * LS + (k == 0 ? 0 : n - k)];
    Yap[(long long)r * WhP + k] = make_float2(0.5f * (z.x + zn.x), 0.5f * (z.y - zn.y));
    Ybp[(long long)r * WhP + k] = make_float2(0.5f * (z.y + zn.y), -0.5f * (z.x - zn.x));
  }
}

// K column pairs per CTA (FS_COL_K for every configured length): Plan16 transforms all 2K lines (forward), Plan8 the first K
// lines (inverse of the mix).
template <class Plan16, class Plan8, int K>
__global__ void __launch_bounds__(FS_COL_T)
fs_cols_kernel(Plan16 plan16, Plan8 plan8, float2* __restrict__ Ya, const float2* __restrict__ Yb,
               const float* __restrict__ lmda, const float2* __restrict__ tw_g, int plane0, int C, int H, int W) {
  constexpr int NL = 2 * K;   // lines per CTA
  extern __shared__ float2 smem[];
  const int n = plan16.n();
  const int m = plan16.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* buf0 = tw + m;
  float2* buf1 = Plan16::kInPlace ? buf0 : buf0 + NL * LS;
  H = n;
  const int Wh = W / 2 + 1;
  const int WhP = (Wh + 7) & ~7;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const float lam = __ldg(lmda + plane / C);
  const int k0 = blockIdx.x * K;
  const int ncols = min(K, Wh - k0);
  for (int t = threadIdx.x; t < m; t += FS_COL_T) tw[t] = __ldg(tw_g + t);
  float2* Yap = Ya + (long long)pl * H * WhP;
  const float2* Ybp = Yb + (long long)pl * H * WhP;
  for (int t = threadIdx.x; t < H * NL; t += FS_COL_T) {
    const int r = t / NL, l = t - r * NL;
    const int cc = l & (K - 1);
    if (cc < ncols) ud_cp_async8(&buf0[l * LS + r], (l < K ? Yap : Ybp) + (long long)r * WhP + k0 + cc);
    else buf0[l * LS + r] = make_float2(0.f, 0.f);
  }
  ud_cp_async_commit();
  ud_cp_async_wait_all();
  __syncthreads();
  float2* res = plan16.run(buf0, buf1, tw, NL, LS);
  // mix in place into lines [0, K) of buf0 (swapped for the inverse transform)
  for (int t = threadIdx.x; t < K * H; t += FS_COL_T) {
    const int cc = t / H, j = t - cc * H;
    const float2 fa = res[cc * LS + j];
    const float2 fb = res[(K + cc) * LS + j];
    const float am = sqrtf(fa.x * fa.x + fa.y * fa.y);
    const float bm = sqrtf(fb.x * fb.x + fb.y * fb.y);
    const float m = lam * am + (1.f - lam) * bm;
    float2 o;
    if (am > 0.f) {
      const float s = m / am;
      o = make_float2(fa.x * s, fa.y * s);
    } else {
      o = make_float2(m, 0.f);   // angle(0) = 0
    }
    res[cc * LS + j] = make_float2(o.y, o.x);   // each thread rewrites only the bin it read: no hazard
  }
  __syncthreads();
  // when the forward plan ping-ponged, `res` may be buf1: run the inverse from there
  float2* other = (res == buf0) ? buf1 : buf0;
  float2* inv = plan8.run(res, other, tw, K, LS);
  for (int t = threadIdx.x; t < H * K; t += FS_COL_T) {
    const int r = t / K, cc = t - r * K;
    if (cc < ncols) {
      const float2 v = inv[cc * LS + r];
      Yap[(long long)r * WhP + k0 + cc] = make_float2(v.y, v.x);   // T overwrites the content spectrum rows
    }
  }
}

template <class Plan, int L>
__global__ void __launch_bounds__(FS_ROW_T)
fs_rows_inv_kernel(Plan plan, const float2* __restrict__ T, float* __restrict__ out, const float2* __restrict__ tw_g,
                   int plane0, int H, int W, float scale) {
  extern __shared__ float2 smem[];
  const int n = plan.n();
  const int m = plan.line_len();     // == n except for Bluestein plans
  const int LS = m | 1;
  float2* tw = smem;
  float2* buf0 = tw + m;
  float2* buf1 = Plan::kInPlace ? buf0 : buf0 + L * LS;
  W = n;
  const int Wh = n / 2 + 1;
  const int WhP = (Wh + 7) & ~7;
  const int pl = blockIdx.y;
  const long long plane = plane0 + pl;
  const int r0 = blockIdx.x * (2 * L);
  for (int t = threadIdx.x; t < m; t += FS_ROW_T) tw[t] = __ldg(tw_g + t);
  const float2* Tp = T + (long long)pl * H * WhP;
  // X_full[k] = T[k] (k < Wh, imaginary parts of self-paired bins dropped), X_full[n-k] = conj T[k];
  // V = Xa + i Xb, stored swapped for the inverse transform.
  for (int t = threadIdx.x; t < L * Wh; t += FS_ROW_T) {
    const int p = t / Wh, k = t - p * Wh;
    const int ra = r0 + 2 * p;
    float2 ta = make_float2(0.f, 0.f), tb = make_float2(0.f, 0.f);
    if (ra < H) ta = Tp[(long long)ra * WhP + k];
    if (ra + 1 < H) tb = Tp[(long long)(ra + 1) * WhP + k];
    float2* line = buf0 + p * LS;
    if ((k == 0) || (2 * k == n)) {
      line[k] = make_float2(tb.x, ta.x);
    } else {
      line[k] = make_float2(ta.y + tb.x, ta.x - tb.y);          // V[k]   = (ar - bi, ai + br) swapped
      line[n - k] = make_float2(tb.x - ta.y, ta.x + tb.y);      // V[n-k] = (ar + bi, br - ai) swapped
    }
  }
  __syncthreads();
  float2* res = plan.run(buf0, buf1, tw, L, LS);   // res[p][c] = (y_b[c], y_a[c])
  float* op = out + plane * (long long)H * W;
  for (int p = 0; p < L; ++p) {
    const int ra = r0 + 2 * p;
    if (ra >= H) break;
    const bool has_b = ra + 1 < H;
    for (int c = threadIdx.x; c < W; c += FS_ROW_T) {
      const float2 v = res[p * LS + c];
      op[(long long)ra * W + c] = v.y * scale;
      if (has_b) op[(long long)(ra + 1) * W + c] = v.x * scale;
    }
  }
}

static size_t fs_smem(int n, int m, int L) {
  return sizeof(float2) * ((size_t)m + (ud_fft_configured(n) ? 1 : 2) * (size_t)L * (m | 1));
}
// Lines per CTA of the rows kernels (FS_ROW_L, /2 or /4) and column pairs per CTA of the cols kernel (FS_COL_K, /2 or
// /4): the most whose two line buffers fit in shared memory, 0 when none does.  The in-place plans of the configured
// lengths always fit.
static int fs_row_lines(int W) {
  if (ud_fft_configured(W)) return FS_ROW_L;
  const int m = ud_any_line_len(W);
  return ud_halving_lines(ud_any_lines(m, sizeof(float2) * (size_t)m, 0, UD_SMEM_CTA_MAX, FS_ROW_L), FS_ROW_L);
}
static int fs_col_k(int H) {
  if (ud_fft_configured(H)) return FS_COL_K;
  const int m = ud_any_line_len(H);
  return ud_halving_lines(ud_any_lines(m, sizeof(float2) * (size_t)m, 0, UD_SMEM_CTA_MAX, FS_COL_L), FS_COL_L) / 2;
}

// Runs launch(plan, lines) with W's row plan and lines per CTA (a std::integral_constant): the configured length's
// in-place plan at FS_ROW_L lines, or the run-time plan at LR lines (FS_ROW_L, /2 or /4).
template <class F>
static int fs_rows_run(int W, int LR, F launch) {
  UD_FFT_CONFIGURED(W, CFG, {
      UdAnyPlan p;
      if (!ud_make_any_plan(W, &p)) return UD_ERR_UNSUPPORTED;
      UD_LINES_DISPATCH(LR, FS_ROW_L, LV, return launch(p, std::integral_constant<int, LV>()));
    }, return launch(CFG::IP<FS_ROW_L, FS_ROW_T>(), std::integral_constant<int, FS_ROW_L>()));
}

static int fs_chunk(int N, int C, int H, int W) {
  const size_t per = 2ull * C * H * fs_whp(W) * sizeof(float2);
  int chunk = (int)((64ull << 20) / (per ? per : 1));
  if (chunk < 1) chunk = 1;
  if (chunk > N) chunk = N;
  if (chunk * C > 65535) chunk = 65535 / C;
  return chunk;
}

extern "C" size_t ud_freq_style_workspace_bytes(int N, int C, int H, int W) {
  return 2ull * (size_t)fs_chunk(N, C, H, W) * C * H * fs_whp(W) * sizeof(float2) + 256;
}

extern "C" int ud_freq_style_transfer(const float* content, const float* style, const float* lmda, float* out, void* ws,
                                      size_t ws_bytes, int N, int C, int H, int W, cudaStream_t stream) {
  UD_REQUIRE(N >= 0 && C >= 1 && H >= 1 && W >= 1, UD_ERR_INVALID, "freq_style: bad shape N=%d C=%d H=%d W=%d", N, C, H, W);
  UD_REQUIRE(H <= UD_FFT_MAX_N && W <= UD_FFT_MAX_N, UD_ERR_UNSUPPORTED, "freq_style: FFT size %dx%d unsupported (n <= %d)",
             H, W, UD_FFT_MAX_N);
  const int LR = fs_row_lines(W), KC = fs_col_k(H);
  UD_REQUIRE(LR > 0, UD_ERR_UNSUPPORTED, "freq_style: %d-point rows do not fit shared memory", W);
  UD_REQUIRE(KC > 0, UD_ERR_UNSUPPORTED, "freq_style: %d-point columns do not fit shared memory", H);
  if (N == 0) return UD_OK;
  UD_REQUIRE(content && style && lmda && out && ws, UD_ERR_INVALID, "freq_style: null pointer");
  UD_REQUIRE(ws_bytes >= ud_freq_style_workspace_bytes(N, C, H, W), UD_ERR_WORKSPACE, "freq_style: workspace too small");
  const int chunk = fs_chunk(N, C, H, W);
  const int Wh = W / 2 + 1;
  float2* Ya = reinterpret_cast<float2*>(ws);
  float2* Yb = Ya + (size_t)chunk * C * H * fs_whp(W);
  const int mW = ud_any_line_len(W), mH = ud_any_line_len(H);
  const float2* twW = ud_twiddles(mW);
  const float2* twH = ud_twiddles(mH);
  if (!twW || !twH) return UD_ERR_CUDA;
  const size_t smR = fs_smem(W, mW, LR), smC = fs_smem(H, mH, 2 * KC);
  const float scale = 1.f / ((float)H * (float)W);
  int rc;
  for (int s0 = 0; s0 < N; s0 += chunk) {
    const int ns = (N - s0 < chunk) ? (N - s0) : chunk;
    const int planes = ns * C, plane0 = s0 * C;
    rc = fs_rows_run(W, LR, [&](auto plan, auto lines) {
      auto k = fs_rows_fwd_kernel<decltype(plan), decltype(lines)::value>;
      const int e = ud_set_smem(k, smR, "freq_style");
      if (e == UD_OK)
        k<<<dim3(ud_cdiv(H, lines), planes), FS_ROW_T, smR, stream>>>(plan, content, style, Ya, Yb, twW, plane0, H, W);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("fs_rows_fwd")) != UD_OK) return rc;
    auto cols = [&](auto p16, auto p8, auto kc) {
      auto k = fs_cols_kernel<decltype(p16), decltype(p8), decltype(kc)::value>;
      const int e = ud_set_smem(k, smC, "freq_style");
      if (e == UD_OK)
        k<<<dim3(ud_cdiv(Wh, kc), planes), FS_COL_T, smC, stream>>>(p16, p8, Ya, Yb, lmda, twH, plane0, C, H, W);
      return e;
    };
    UD_FFT_CONFIGURED(H, CFG, {
        UdAnyPlan p;
        if (!ud_make_any_plan(H, &p)) return UD_ERR_UNSUPPORTED;
        UD_LINES_DISPATCH(KC, FS_COL_K, KV, rc = cols(p, p, std::integral_constant<int, KV>()));
      }, rc = cols(CFG::IP<FS_COL_L, FS_COL_T>(), CFG::IP<FS_COL_K, FS_COL_T>(), std::integral_constant<int, FS_COL_K>()));
    if (rc != UD_OK || (rc = ud_check_launch("fs_cols")) != UD_OK) return rc;
    rc = fs_rows_run(W, LR, [&](auto plan, auto lines) {
      auto k = fs_rows_inv_kernel<decltype(plan), decltype(lines)::value>;
      const int e = ud_set_smem(k, smR, "freq_style");
      if (e == UD_OK)
        k<<<dim3(ud_cdiv(H, 2 * lines), planes), FS_ROW_T, smR, stream>>>(plan, Ya, out, twW, plane0, H, W, scale);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("fs_rows_inv")) != UD_OK) return rc;
  }
  return UD_OK;
}
