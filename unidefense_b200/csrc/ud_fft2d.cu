// Generic batched 2-D real FFT pair in the reference's cat([re, im], dim=1) layout           (SURVEY.md §8b)
//
//   ud_rfft2 :  x [N,C,h,w]  ->  xf [N,2C,h,w/2+1]  = cat([re, im], 1) of torch.fft.rfft2(x, norm)
//   ud_irfft2:  xf [N,2C,h,w/2+1] (optionally * mask [N,h*(w/2+1)])  ->  y [N,C,h,w] = torch.fft.irfft2(.., s=(h,w))
// plus the two autograd adjoints (fft_c2r_backward / fft_r2c_backward, SURVEY App. B.2/B.3) selected by a flag, for
// ANY 1 <= h, w <= UD_FFT_MAX_N: mixed radix when every prime factor is <= 23, Bluestein otherwise
// (ud_fft_any.cuh).  Reference call sites: model/unidefense.py:135-145 (feature maps), :246-249 (images),
// model/modules.py:43-54, model/efficientnet/exp.py:55-65, model/resnet/exp.py:44-54 (SFConv).
// Planes with h, w <= 64 take the one-CTA-per-plane path of ud_attention.cu (no workspace); everything else runs
// rows and columns as two kernels through a caller-provided workspace T [planes][h][w/2+1] complex:
//   r2c:  rows (two real rows packed into one complex line, unpacked on store)  ->  T  ->  columns, scale, planar store
//   c2r:  columns (inverse, swap trick; mask and column multipliers applied on load)  ->  T  ->  rows: the half
//         spectrum is zero-padded to w points and the real part of the inverse transform kept -- exactly
//         y[r][c] = sum_k m_k Re(U[r][k] e^{+2 pi i k c / w}) (the imaginary parts of the DC / Nyquist columns drop
//         out as they do in pocketfft / cuFFT C2R).
// Each CTA keeps L lines in shared memory (L chosen so the two ping-pong buffers fit in ~96 KB) and runs the
// Stockham stages over all of them; global accesses are row segments of L (columns) or w (rows) consecutive elements.
#include "../../include/unidefense_b200.h"
#include "ud_fft_any.cuh"

#define F2_THREADS 256
#define F2_MAX_GRID_Y 65535

int ud_rfft2_small(const float* x, float* xf, int N, int C, int h, int w, int norm_ortho, int adjoint_of_inverse,
                   cudaStream_t stream);
int ud_irfft2_small(const float* xf, const float* mask, float* y, int N, int C, int h, int w, int norm_ortho,
                    int adjoint_of_forward, cudaStream_t stream);
bool ud_fft2_small_ok(int h, int w);

static int f2_lines(const UdAnyPlan& p) {
  const int L = ud_any_lines(p.m, 0, 0, 96u << 10, 16);   // 96 KB of line buffers (the twiddles come on top)
  return L < 1 ? 1 : L;
}
static size_t f2_smem(const UdAnyPlan& p, int L) {
  return sizeof(float2) * ((size_t)p.m + 2ull * L * ud_any_line_stride(p));
}

// Plans: UdAnyPlan (any size, run time) or the in-place static plans of the configured image sizes (every index
// constant-folded; F2_L lines per CTA, F2_THREADS threads).  `tw_g` = exp(-2 pi i t / m), t < m = plan.line_len().
#define F2_L 16
template <class Plan>
__device__ __forceinline__ void f2_stage_tw(float2* tw_s, const Plan& p, const float2* __restrict__ tw_g) {
  for (int t = threadIdx.x; t < p.line_len(); t += blockDim.x) tw_s[t] = __ldg(tw_g + t);
}

// rows of the forward transform: line l = rows (2p, 2p+1) of the plane packed as a + i b
template <class Plan>
__global__ void __launch_bounds__(F2_THREADS)
f2_rows_r2c_kernel(Plan plan, const float2* __restrict__ tw_g, const float* __restrict__ x, float2* __restrict__ T, int h, int w, int L,
                   int plane0) {
  extern __shared__ float2 f2sm[];
  const int LS = plan.line_len() | 1, wh = w / 2 + 1;
  float2* tw_s = f2sm;
  float2* a = tw_s + plan.line_len();
  float2* b = a + L * LS;
  const long long plane = (long long)plane0 + blockIdx.y;
  const int p0 = blockIdx.x * L;                      // first row pair of this CTA
  const float* xp = x + plane * (long long)h * w;
  f2_stage_tw(tw_s, plan, tw_g);
  for (int idx = threadIdx.x; idx < L * w; idx += blockDim.x) {
    const int l = idx / w, j = idx - l * w;
    const int r = 2 * (p0 + l);
    a[l * LS + j] = make_float2(r < h ? __ldg(xp + (long long)r * w + j) : 0.f,
                                r + 1 < h ? __ldg(xp + (long long)(r + 1) * w + j) : 0.f);
  }
  __syncthreads();
  const float2* res = plan.run(a, b, tw_s, L, LS);
  float2* Tp = T + plane * (long long)h * wh;
  for (int idx = threadIdx.x; idx < L * wh; idx += blockDim.x) {
    const int l = idx / wh, k = idx - l * wh;
    const int r = 2 * (p0 + l);
    if (r >= h) continue;
    const float2 z1 = res[l * LS + k], z2 = res[l * LS + (k == 0 ? 0 : w - k)];
    // A[k] = (Z[k] + conj Z[w-k]) / 2,  B[k] = (Z[k] - conj Z[w-k]) / 2i
    Tp[(long long)r * wh + k] = make_float2(0.5f * (z1.x + z2.x), 0.5f * (z1.y - z2.y));
    if (r + 1 < h) Tp[(long long)(r + 1) * wh + k] = make_float2(0.5f * (z1.y + z2.y), -0.5f * (z1.x - z2.x));
  }
}

// columns of the forward transform: line l = column k0 + l of T; planar store with scale and column multipliers
template <class Plan>
__global__ void __launch_bounds__(F2_THREADS)
f2_cols_fwd_kernel(Plan plan, const float2* __restrict__ tw_g, const float2* __restrict__ T, float* __restrict__ out, int C, int h, int w, int L,
                   float scale, int colmul, int plane0) {
  extern __shared__ float2 f2sm[];
  const int LS = plan.line_len() | 1, wh = w / 2 + 1;
  float2* tw_s = f2sm;
  float2* a = tw_s + plan.line_len();
  float2* b = a + L * LS;
  const long long plane = (long long)plane0 + blockIdx.y;
  const int k0 = blockIdx.x * L;
  const float2* Tp = T + plane * (long long)h * wh;
  f2_stage_tw(tw_s, plan, tw_g);
  for (int idx = threadIdx.x; idx < L * h; idx += blockDim.x) {
    const int r = idx / L, l = idx - r * L;
    a[l * LS + r] = (k0 + l < wh) ? __ldg(Tp + (long long)r * wh + k0 + l) : make_float2(0.f, 0.f);
  }
  __syncthreads();
  const float2* res = plan.run(a, b, tw_s, L, LS);
  const long long n = plane / C, c = plane - n * C;
  float* ore = out + (n * 2 * C + c) * (long long)h * wh;
  float* oim = out + (n * 2 * C + C + c) * (long long)h * wh;
  const int last = (w % 2 == 0) ? wh - 1 : wh;
  for (int idx = threadIdx.x; idx < L * h; idx += blockDim.x) {
    const int r = idx / L, l = idx - r * L;
    const int k = k0 + l;
    if (k >= wh) continue;
    const float s = (colmul && k >= 1 && k < last) ? 2.f * scale : scale;
    const float2 v = res[l * LS + r];
    ore[(long long)r * wh + k] = v.x * s;
    oim[(long long)r * wh + k] = v.y * s;
  }
}

// columns of the inverse transform: U[r][k] = sum_j m_k Z[j][k] e^{+2 pi i j r / h}  (unnormalised)
template <class Plan>
__global__ void __launch_bounds__(F2_THREADS)
f2_cols_inv_kernel(Plan plan, const float2* __restrict__ tw_g, const float* __restrict__ in, const float* __restrict__ mask, float2* __restrict__ T,
                   int C, int h, int w, int L, int colmul, int plane0) {
  extern __shared__ float2 f2sm[];
  const int LS = plan.line_len() | 1, wh = w / 2 + 1;
  float2* tw_s = f2sm;
  float2* a = tw_s + plan.line_len();
  float2* b = a + L * LS;
  const long long plane = (long long)plane0 + blockIdx.y;
  const int k0 = blockIdx.x * L;
  const long long n = plane / C, c = plane - n * C;
  const float* ire = in + (n * 2 * C + c) * (long long)h * wh;
  const float* iim = in + (n * 2 * C + C + c) * (long long)h * wh;
  const float* mk = mask ? mask + n * (long long)h * wh : nullptr;
  const int last = (w % 2 == 0) ? wh - 1 : wh;
  f2_stage_tw(tw_s, plan, tw_g);
  for (int idx = threadIdx.x; idx < L * h; idx += blockDim.x) {
    const int r = idx / L, l = idx - r * L;
    const int k = k0 + l;
    float2 v = make_float2(0.f, 0.f);
    if (k < wh) {
      const long long o = (long long)r * wh + k;
      float m = mk ? __ldg(mk + o) : 1.f;
      if (colmul && k >= 1 && k < last) m *= 2.f;
      v = make_float2(__ldg(iim + o) * m, __ldg(ire + o) * m);          // swapped: IFFT(z) = swap(FFT(swap(z)))
    }
    a[l * LS + r] = v;
  }
  __syncthreads();
  const float2* res = plan.run(a, b, tw_s, L, LS);
  float2* Tp = T + plane * (long long)h * wh;
  for (int idx = threadIdx.x; idx < L * h; idx += blockDim.x) {
    const int r = idx / L, l = idx - r * L;
    if (k0 + l >= wh) continue;
    const float2 v = res[l * LS + r];
    Tp[(long long)r * wh + k0 + l] = make_float2(v.y, v.x);
  }
}

// rows of the inverse transform: y[r][c] = scale * Re sum_{k < wh} U[r][k] e^{+2 pi i k c / w}
template <class Plan>
__global__ void __launch_bounds__(F2_THREADS)
f2_rows_c2r_kernel(Plan plan, const float2* __restrict__ tw_g, const float2* __restrict__ T, float* __restrict__ y, int h, int w, int L, float scale,
                   int plane0) {
  extern __shared__ float2 f2sm[];
  const int LS = plan.line_len() | 1, wh = w / 2 + 1;
  float2* tw_s = f2sm;
  float2* a = tw_s + plan.line_len();
  float2* b = a + L * LS;
  const long long plane = (long long)plane0 + blockIdx.y;
  const int r0 = blockIdx.x * L;
  const float2* Tp = T + plane * (long long)h * wh;
  f2_stage_tw(tw_s, plan, tw_g);
  for (int idx = threadIdx.x; idx < L * w; idx += blockDim.x) {
    const int l = idx / w, k = idx - l * w;
    float2 v = make_float2(0.f, 0.f);
    if (r0 + l < h && k < wh) {
      const float2 u = __ldg(Tp + (long long)(r0 + l) * wh + k);
      v = make_float2(u.y, u.x);                                         // swapped
    }
    a[l * LS + k] = v;
  }
  __syncthreads();
  const float2* res = plan.run(a, b, tw_s, L, LS);
  float* yp = y + plane * (long long)h * w;
  for (int idx = threadIdx.x; idx < L * w; idx += blockDim.x) {
    const int l = idx / w, cc = idx - l * w;
    if (r0 + l < h) yp[(long long)(r0 + l) * w + cc] = res[l * LS + cc].y * scale;   // Re of the unswapped result
  }
}

// Runs launch(plan, L) with n's plan: the configured length's in-place plan at F2_L lines per CTA, or the run-time
// plan `any` (m = n for every configured length, so both share f2_smem).
template <class F>
static int f2_run(int n, const UdAnyPlan& any, F launch) {
  UD_FFT_CONFIGURED(n, CFG, return launch(any, f2_lines(any)), return launch(CFG::IP<F2_L, F2_THREADS>(), F2_L));
}

static float f2_scale(int h, int w, int norm_ortho, bool inverse) {
  if (norm_ortho) return 1.f / sqrtf((float)h * (float)w);
  return inverse ? 1.f / ((float)h * (float)w) : 1.f;
}

static int f2_check(const char* what, int N, int C, int h, int w) {
  UD_REQUIRE(N >= 0 && C >= 1 && h >= 1 && w >= 1, UD_ERR_INVALID, "%s: bad shape N=%d C=%d h=%d w=%d", what, N, C, h, w);
  UD_REQUIRE(h <= UD_FFT_MAX_N && w <= UD_FFT_MAX_N, UD_ERR_UNSUPPORTED, "%s: plane %dx%d exceeds UD_FFT_MAX_N=%d", what,
             h, w, UD_FFT_MAX_N);
  UD_REQUIRE((long long)N * C <= 0x7fffffffLL, UD_ERR_UNSUPPORTED, "%s: too many planes", what);
  return UD_OK;
}

extern "C" size_t ud_rfft2_workspace_bytes(int N, int C, int h, int w) {
  if (N <= 0 || C <= 0 || h <= 0 || w <= 0 || ud_fft2_small_ok(h, w)) return 0;
  return sizeof(float2) * (size_t)N * C * h * (w / 2 + 1);
}

extern "C" int ud_rfft2(const float* x, float* xf, void* ws, size_t ws_bytes, int N, int C, int h, int w, int norm_ortho,
                        int adjoint_of_inverse, cudaStream_t stream) {
  int rc = f2_check("rfft2", N, C, h, w);
  if (rc != UD_OK) return rc;
  if (N == 0) return UD_OK;
  UD_REQUIRE(x && xf, UD_ERR_INVALID, "rfft2: null pointer");
  if (ud_fft2_small_ok(h, w)) return ud_rfft2_small(x, xf, N, C, h, w, norm_ortho, adjoint_of_inverse, stream);
  UD_REQUIRE(ws && ws_bytes >= ud_rfft2_workspace_bytes(N, C, h, w), UD_ERR_WORKSPACE, "rfft2: workspace too small");
  UdAnyPlan pw, ph;
  if (!ud_make_any_plan(w, &pw) || !ud_make_any_plan(h, &ph)) return UD_ERR_UNSUPPORTED;
  float2* T = static_cast<float2*>(ws);
  const int planes = N * C, wh = w / 2 + 1;
  const float scale = f2_scale(h, w, norm_ortho, adjoint_of_inverse != 0);
  for (int p0 = 0; p0 < planes; p0 += F2_MAX_GRID_Y) {            // gridDim.y <= 65535
    const int np = planes - p0 < F2_MAX_GRID_Y ? planes - p0 : F2_MAX_GRID_Y;
    rc = f2_run(w, pw, [&](auto pl, int L) {
      auto k = f2_rows_r2c_kernel<decltype(pl)>;
      const size_t sm = f2_smem(pw, L);
      const int e = ud_set_smem(k, sm, "fft2");
      if (e == UD_OK) k<<<dim3(ud_cdiv((h + 1) / 2, L), np), F2_THREADS, sm, stream>>>(pl, pw.tw, x, T, h, w, L, p0);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("rfft2_rows")) != UD_OK) return rc;
    rc = f2_run(h, ph, [&](auto pl, int L) {
      auto k = f2_cols_fwd_kernel<decltype(pl)>;
      const size_t sm = f2_smem(ph, L);
      const int e = ud_set_smem(k, sm, "fft2");
      if (e == UD_OK)
        k<<<dim3(ud_cdiv(wh, L), np), F2_THREADS, sm, stream>>>(pl, ph.tw, T, xf, C, h, w, L, scale, adjoint_of_inverse, p0);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("rfft2_cols")) != UD_OK) return rc;
  }
  return UD_OK;
}

extern "C" int ud_irfft2(const float* xf, const float* mask, float* y, void* ws, size_t ws_bytes, int N, int C, int h,
                         int w, int norm_ortho, int adjoint_of_forward, cudaStream_t stream) {
  int rc = f2_check("irfft2", N, C, h, w);
  if (rc != UD_OK) return rc;
  if (N == 0) return UD_OK;
  UD_REQUIRE(xf && y, UD_ERR_INVALID, "irfft2: null pointer");
  if (ud_fft2_small_ok(h, w)) return ud_irfft2_small(xf, mask, y, N, C, h, w, norm_ortho, adjoint_of_forward, stream);
  UD_REQUIRE(ws && ws_bytes >= ud_rfft2_workspace_bytes(N, C, h, w), UD_ERR_WORKSPACE, "irfft2: workspace too small");
  UdAnyPlan pw, ph;
  if (!ud_make_any_plan(w, &pw) || !ud_make_any_plan(h, &ph)) return UD_ERR_UNSUPPORTED;
  float2* T = static_cast<float2*>(ws);
  const int planes = N * C, wh = w / 2 + 1;
  const float scale = f2_scale(h, w, norm_ortho, adjoint_of_forward == 0);
  for (int p0 = 0; p0 < planes; p0 += F2_MAX_GRID_Y) {
    const int np = planes - p0 < F2_MAX_GRID_Y ? planes - p0 : F2_MAX_GRID_Y;
    rc = f2_run(h, ph, [&](auto pl, int L) {
      auto k = f2_cols_inv_kernel<decltype(pl)>;
      const size_t sm = f2_smem(ph, L);
      const int e = ud_set_smem(k, sm, "fft2");
      if (e == UD_OK)
        k<<<dim3(ud_cdiv(wh, L), np), F2_THREADS, sm, stream>>>(pl, ph.tw, xf, mask, T, C, h, w, L, adjoint_of_forward ? 0 : 1, p0);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("irfft2_cols")) != UD_OK) return rc;
    rc = f2_run(w, pw, [&](auto pl, int L) {
      auto k = f2_rows_c2r_kernel<decltype(pl)>;
      const size_t sm = f2_smem(pw, L);
      const int e = ud_set_smem(k, sm, "fft2");
      if (e == UD_OK) k<<<dim3(ud_cdiv(h, L), np), F2_THREADS, sm, stream>>>(pl, pw.tw, T, y, h, w, L, scale, p0);
      return e;
    });
    if (rc != UD_OK || (rc = ud_check_launch("irfft2_rows")) != UD_OK) return rc;
  }
  return UD_OK;
}
