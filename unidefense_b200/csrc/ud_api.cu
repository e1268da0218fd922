// Library-wide state for libunidefense_b200.so: thread-local error string, version, the
// per-(device, n) twiddle-table cache and FFT plan factorisation.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/unidefense_b200.h"
#include "ud_fft.cuh"
#include "ud_fft_any.cuh"

static thread_local char g_err[512] = "";

void ud_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void ud_count_launch(void) { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" long long ud_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int ud_check_launch(const char* what) {
  ud_count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ud_set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e));
    return UD_ERR_CUDA;
  }
  return UD_OK;
}

extern "C" const char* ud_last_error(void) { return g_err; }
extern "C" int ud_version(void) { return UD_B200_VERSION; }

bool ud_make_dyn_plan(int n, UdDynPlan* plan) {
  if (n < 1) return false;
  static const int primes[] = {23, 19, 17, 13, 11, 7, 5, 3};
  plan->n_ = n;
  plan->nstages = 0;
  int m = n;
  for (int p : primes) {
    while (m % p == 0) {
      if (plan->nstages >= UD_FFT_MAX_STAGES) return false;
      plan->radix[plan->nstages++] = p;
      m /= p;
    }
  }
  while (m % 4 == 0) {
    if (plan->nstages >= UD_FFT_MAX_STAGES) return false;
    plan->radix[plan->nstages++] = 4;
    m /= 4;
  }
  if (m % 2 == 0) {
    if (plan->nstages >= UD_FFT_MAX_STAGES) return false;
    plan->radix[plan->nstages++] = 2;
    m /= 2;
  }
  return m == 1;
}

extern "C" int ud_fft_size_supported(int n) {
  UdDynPlan p;
  return (n >= 1 && n <= UD_FFT_MAX_N && ud_make_dyn_plan(n, &p)) ? 1 : 0;
}
extern "C" int ud_fft_size_any(int n) { return (n >= 1 && n <= UD_FFT_MAX_N) ? 1 : 0; }

// exp(-2 pi i t / n) with exact octant symmetry (so W^(n/4), W^(n/2) ... are exact)
static void twiddle_host(int n, std::vector<float2>& out) {
  out.resize(n);
  for (int t = 0; t < n; ++t) {
    // reduce the angle 2 pi t/n to the first octant using integer arithmetic on 8t/n
    long long num = (long long)t * 8;  // angle = (num/n) * pi/4
    int oct = (int)(num / n);
    long long rem = num - (long long)oct * n;  // in [0, n): fraction of an octant
    double c, s;
    if ((oct & 1) == 0) {
      double a = (double)rem / (double)n * (M_PI / 4.0);
      c = cos(a);
      s = sin(a);
    } else {
      double a = (double)(n - rem) / (double)n * (M_PI / 4.0);
      c = sin(a);
      s = cos(a);
    }
    // now (c,s) = (cos, sin) of the angle folded into [0, pi/2) for quadrant oct/2
    double cr, sr;
    switch ((oct >> 1) & 3) {
      case 0: cr = c; sr = s; break;
      case 1: cr = -s; sr = c; break;
      case 2: cr = -c; sr = -s; break;
      default: cr = s; sr = -c; break;
    }
    if (rem == 0) {  // exact multiples of pi/4: kill rounding residue on the axes
      if ((oct & 1) == 0) {
        const double ex[4][2] = {{1, 0}, {0, 1}, {-1, 0}, {0, -1}};
        cr = ex[(oct >> 1) & 3][0];
        sr = ex[(oct >> 1) & 3][1];
      }
    }
    out[t] = make_float2((float)cr, (float)(-sr));
  }
}

static std::mutex g_tw_mutex;
static std::map<std::pair<int, int>, float2*> g_tw_cache;

const float2* ud_twiddles(int n) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    ud_set_error("cudaGetDevice failed");
    return nullptr;
  }
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto key = std::make_pair(dev, n);
  auto it = g_tw_cache.find(key);
  if (it != g_tw_cache.end()) return it->second;
  std::vector<float2> h;
  twiddle_host(n, h);
  float2* d = nullptr;
  if (cudaMalloc(&d, sizeof(float2) * (size_t)n) != cudaSuccess) {
    ud_set_error("cudaMalloc(twiddles n=%d) failed", n);
    return nullptr;
  }
  // synchronous copy on the legacy stream: tables are immutable afterwards, and any stream
  // that later reads them is ordered after this call returns.
  if (cudaMemcpy(d, h.data(), sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice) != cudaSuccess) {
    ud_set_error("cudaMemcpy(twiddles n=%d) failed", n);
    cudaFree(d);
    return nullptr;
  }
  g_tw_cache[key] = d;
  return d;
}

static std::map<std::pair<int, std::pair<int, int>>, float2*> g_lerp_cache;

const float2* ud_lerp_table(int in, int out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    ud_set_error("cudaGetDevice failed");
    return nullptr;
  }
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto key = std::make_pair(dev, std::make_pair(in, out));
  auto it = g_lerp_cache.find(key);
  if (it != g_lerp_cache.end()) return it->second;
  std::vector<float2> h((size_t)out);
  const float scale = ud_ac_scale(in, out);
  for (int d = 0; d < out; ++d) {
    const float src = scale * (float)d;       // ATen: area_pixel_compute_source_index, align_corners=True
    const int i0 = (int)src;
    union { int i; float f; } u;
    u.i = i0;
    h[d] = make_float2(u.f, src - (float)i0);
  }
  float2* p = nullptr;
  if (cudaMalloc(&p, sizeof(float2) * (size_t)out) != cudaSuccess) {
    ud_set_error("cudaMalloc(lerp table %d->%d) failed", in, out);
    return nullptr;
  }
  if (cudaMemcpy(p, h.data(), sizeof(float2) * (size_t)out, cudaMemcpyHostToDevice) != cudaSuccess) {
    ud_set_error("cudaMemcpy(lerp table %d->%d) failed", in, out);
    cudaFree(p);
    return nullptr;
  }
  g_lerp_cache[key] = p;
  return p;
}

static std::map<std::pair<int, std::pair<int, int>>, int2*> g_range_cache;

const int2* ud_lerp_ranges(int in, int out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    ud_set_error("cudaGetDevice failed");
    return nullptr;
  }
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto key = std::make_pair(dev, std::make_pair(in, out));
  auto it = g_range_cache.find(key);
  if (it != g_range_cache.end()) return it->second;
  std::vector<int2> h((size_t)in, make_int2(out, -1));
  const float scale = ud_ac_scale(in, out);
  for (int d = 0; d < out; ++d) {
    const float src = scale * (float)d;
    const int i0 = (int)src;
    const int i1 = i0 + ((i0 < in - 1) ? 1 : 0);
    for (int i : {i0, i1}) {
      if (d < h[i].x) h[i].x = d;
      if (d > h[i].y) h[i].y = d;
    }
  }
  int2* p = nullptr;
  if (cudaMalloc(&p, sizeof(int2) * (size_t)in) != cudaSuccess) {
    ud_set_error("cudaMalloc(lerp ranges %d->%d) failed", in, out);
    return nullptr;
  }
  if (cudaMemcpy(p, h.data(), sizeof(int2) * (size_t)in, cudaMemcpyHostToDevice) != cudaSuccess) {
    ud_set_error("cudaMemcpy(lerp ranges %d->%d) failed", in, out);
    cudaFree(p);
    return nullptr;
  }
  g_range_cache[key] = p;
  return p;
}


// ---- Bluestein tables (ud_fft_any.cuh) -------------------------------------------------------------
struct BluesteinTables {
  float2* chirp;
  float2* bhat;
};
static std::map<std::pair<int, int>, BluesteinTables> g_bs_cache;

// in-place radix-2 FFT in double precision (host, table construction only)
static void host_fft_pow2(std::vector<double>& re, std::vector<double>& im) {
  const size_t m = re.size();
  for (size_t i = 1, j = 0; i < m; ++i) {
    size_t bit = m >> 1;
    for (; j & bit; bit >>= 1) j ^= bit;
    j ^= bit;
    if (i < j) {
      std::swap(re[i], re[j]);
      std::swap(im[i], im[j]);
    }
  }
  for (size_t len = 2; len <= m; len <<= 1) {
    for (size_t i = 0; i < m; i += len) {
      for (size_t k = 0; k < len / 2; ++k) {
        const double ang = -2.0 * M_PI * (double)k / (double)len;
        const double wr = cos(ang), wi = sin(ang);
        const size_t a = i + k, b = i + k + len / 2;
        const double xr = re[b] * wr - im[b] * wi, xi = re[b] * wi + im[b] * wr;
        re[b] = re[a] - xr;
        im[b] = im[a] - xi;
        re[a] += xr;
        im[a] += xi;
      }
    }
  }
}

int ud_any_line_len(int n) {
  if (n < 1 || n > UD_FFT_MAX_N) return 0;
  UdDynPlan p;
  if (ud_make_dyn_plan(n, &p)) return n;
  int m = 1;
  while (m < 2 * n - 1) m <<= 1;
  return m;
}

bool ud_make_any_plan(int n, UdAnyPlan* plan) {
  if (n < 1 || n > UD_FFT_MAX_N) {
    ud_set_error("FFT size %d outside [1, %d]", n, UD_FFT_MAX_N);
    return false;
  }
  plan->n_ = n;
  plan->chirp = nullptr;
  plan->bhat = nullptr;
  if (ud_make_dyn_plan(n, &plan->inner)) {
    plan->m = n;
    plan->bluestein = 0;
    plan->tw = ud_twiddles(n);
    return plan->tw != nullptr;
  }
  const int m = ud_any_line_len(n);
  plan->m = m;
  plan->bluestein = 1;
  if (!ud_make_dyn_plan(m, &plan->inner)) {
    ud_set_error("FFT size %d: no stage plan for the Bluestein length %d", n, m);
    return false;
  }
  plan->tw = ud_twiddles(m);
  if (!plan->tw) return false;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    ud_set_error("cudaGetDevice failed");
    return false;
  }
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto key = std::make_pair(dev, n);
  auto it = g_bs_cache.find(key);
  if (it == g_bs_cache.end()) {
    std::vector<double> wr(n), wi(n), br(m, 0.0), bi(m, 0.0);
    for (int j = 0; j < n; ++j) {
      const long long q = ((long long)j * j) % (2LL * n);      // phase pi * j^2 / n reduced mod 2 pi
      const double ang = M_PI * (double)q / (double)n;
      wr[j] = cos(ang);
      wi[j] = -sin(ang);                                       // w[j] = exp(-i pi j^2 / n)
    }
    for (int t = 0; t < n; ++t) {                              // conj(w), even in t, wrapped to length m
      br[t] = wr[t];
      bi[t] = -wi[t];
      if (t) {
        br[m - t] = wr[t];
        bi[m - t] = -wi[t];
      }
    }
    host_fft_pow2(br, bi);
    std::vector<float2> hc(n), hb(m);
    for (int j = 0; j < n; ++j) hc[j] = make_float2((float)wr[j], (float)wi[j]);
    for (int k = 0; k < m; ++k) hb[k] = make_float2((float)(br[k] / m), (float)(bi[k] / m));
    BluesteinTables t = {nullptr, nullptr};
    if (cudaMalloc(&t.chirp, sizeof(float2) * (size_t)n) != cudaSuccess ||
        cudaMalloc(&t.bhat, sizeof(float2) * (size_t)m) != cudaSuccess ||
        cudaMemcpy(t.chirp, hc.data(), sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(t.bhat, hb.data(), sizeof(float2) * (size_t)m, cudaMemcpyHostToDevice) != cudaSuccess) {
      ud_set_error("Bluestein tables for n=%d: allocation or copy failed", n);
      if (t.chirp) cudaFree(t.chirp);
      if (t.bhat) cudaFree(t.bhat);
      return false;
    }
    it = g_bs_cache.emplace(key, t).first;
  }
  plan->chirp = it->second.chirp;
  plan->bhat = it->second.bhat;
  return true;
}
