// a16 -- stencil / resampling perturbations of the second training pass   (SURVEY.md §8a row a16)
//
// Reference: random_blur (model/modules.py:15-16 -> torchvision gaussian_blur, 5x5, sigma 1.1,
// reflect padding, depthwise) and downscale (model/modules.py:19-21: nearest x0.75 then nearest
// back to the input size).  Both are one read + one write of the image; the 25 taps and the
// gather hit L1/L2.  Their adjoints (the input gradient) are gathers too: one fixed-order sum per
// input pixel, no atomics.
#include <math.h>

#include "../../include/unidefense_b200.h"
#include "ud_common.cuh"

struct PtBlurW {
  float k[5];
};

__device__ __forceinline__ int pt_reflect(int i, int n) {
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

// one thread per output pixel; 32x8 tiles keep the 5x5 neighbourhoods in L1
__global__ void __launch_bounds__(256)
pt_blur5_kernel(const float* __restrict__ x, float* __restrict__ y, int H, int W, PtBlurW wy, PtBlurW wx) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (c >= W || r >= H) return;
  const float* p = x + (long long)blockIdx.z * H * W;
  int cc[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) cc[j] = pt_reflect(c + j - 2, W);
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const float* row = p + (long long)pt_reflect(r + i - 2, H) * W;
#pragma unroll
    for (int j = 0; j < 5; ++j) acc = fmaf(wy.k[i] * wx.k[j], __ldg(row + cc[j]), acc);
  }
  y[(long long)blockIdx.z * H * W + (long long)r * W + c] = acc;
}

// torchvision _get_gaussian_kernel1d: sigma = 0.3*((k-1)*0.5-1)+0.8 = 1.1, fp32 arithmetic
static PtBlurW pt_blur_weights() {
  PtBlurW w;
  const float sigma = 0.3f * ((5 - 1) * 0.5f - 1.f) + 0.8f;
  float s = 0.f;
  for (int i = 0; i < 5; ++i) {
    const float t = (float)(i - 2) / sigma;
    w.k[i] = expf(-0.5f * t * t);
    s += w.k[i];
  }
  for (int i = 0; i < 5; ++i) w.k[i] /= s;
  return w;
}

extern "C" int ud_gaussian_blur5(const float* x, float* y, int planes, int H, int W, cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && H >= 3 && W >= 3, UD_ERR_INVALID,
             "gaussian_blur5: bad shape planes=%d H=%d W=%d (reflect padding 2 needs H,W >= 3)", planes, H, W);
  if (planes == 0) return UD_OK;
  UD_REQUIRE(x && y, UD_ERR_INVALID, "gaussian_blur5: null pointer");
  UD_REQUIRE(planes <= 65535, UD_ERR_UNSUPPORTED, "gaussian_blur5: too many planes (%d)", planes);
  const PtBlurW w = pt_blur_weights();
  pt_blur5_kernel<<<dim3(ud_cdiv(W, 32), ud_cdiv(H, 8), planes), 256, 0, stream>>>(x, y, H, W, w, w);
  return ud_check_launch("gaussian_blur5");
}

// Adjoint of the blur: gx[i,j] = sum_{r,c} Ay[i,r] Ax[j,c] gy[r,c] with A[i,r] = sum_t k[t] [reflect(r+t-2) == i].
// Every output row r that reaches input row i lies in [i-2, i+2] (the reflected taps of the two border rows fold back
// inside that window), so the gather is a 5x5 window with border-aware effective weights.
__device__ __forceinline__ float pt_adj_w(const PtBlurW& k, int i, int r, int n) {
  float a = 0.f;
#pragma unroll
  for (int t = 0; t < 5; ++t) a += (pt_reflect(r + t - 2, n) == i) ? k.k[t] : 0.f;
  return a;
}

__global__ void __launch_bounds__(256)
pt_blur5_bwd_kernel(const float* __restrict__ gy, float* __restrict__ gx, int H, int W, PtBlurW wy, PtBlurW wx) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (c >= W || r >= H) return;
  const float* p = gy + (long long)blockIdx.z * H * W;
  float ax[5];
  int cc[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    cc[j] = c + j - 2;
    ax[j] = (cc[j] >= 0 && cc[j] < W) ? pt_adj_w(wx, c, cc[j], W) : 0.f;
    cc[j] = min(max(cc[j], 0), W - 1);
  }
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int rr = r + i - 2;
    if (rr < 0 || rr >= H) continue;
    const float ay = pt_adj_w(wy, r, rr, H);
    const float* row = p + (long long)rr * W;
    float t = 0.f;
#pragma unroll
    for (int j = 0; j < 5; ++j) t = fmaf(ax[j], __ldg(row + cc[j]), t);
    acc = fmaf(ay, t, acc);
  }
  gx[(long long)blockIdx.z * H * W + (long long)r * W + c] = acc;
}

extern "C" int ud_gaussian_blur5_bwd(const float* gy, float* gx, int planes, int H, int W, cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && H >= 3 && W >= 3, UD_ERR_INVALID,
             "gaussian_blur5_bwd: bad shape planes=%d H=%d W=%d (reflect padding 2 needs H,W >= 3)", planes, H, W);
  if (planes == 0) return UD_OK;
  UD_REQUIRE(gy && gx, UD_ERR_INVALID, "gaussian_blur5_bwd: null pointer");
  UD_REQUIRE(planes <= 65535, UD_ERR_UNSUPPORTED, "gaussian_blur5_bwd: too many planes (%d)", planes);
  const PtBlurW w = pt_blur_weights();
  pt_blur5_bwd_kernel<<<dim3(ud_cdiv(W, 32), ud_cdiv(H, 8), planes), 256, 0, stream>>>(gy, gx, H, W, w, w);
  return ud_check_launch("gaussian_blur5_bwd");
}

// ATen nearest: src = min((int)floorf(dst * scale), in - 1), scale fp32.
__global__ void pt_downscale_kernel(const float* __restrict__ x, float* __restrict__ y, long long total, int H, int W,
                                    int h, int w, float sdy, float sdx, float suy, float sux) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % W);
    const long long t = i / W;
    const int r = (int)(t % H);
    const long long plane = t / H;
    const int rm = min((int)floorf((float)r * suy), h - 1);   // row in the low-res image
    const int cm = min((int)floorf((float)c * sux), w - 1);
    const int rs = min((int)floorf((float)rm * sdy), H - 1);  // its source row in the input
    const int cs = min((int)floorf((float)cm * sdx), W - 1);
    y[i] = __ldg(x + plane * (long long)H * W + (long long)rs * W + cs);
  }
}

extern "C" int ud_downscale_nearest(const float* x, float* y, int planes, int H, int W, float bottleneck_scale,
                                    cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && H >= 1 && W >= 1 && bottleneck_scale > 0.f, UD_ERR_INVALID, "downscale: bad arguments");
  const int h = (int)floor((double)H * (double)bottleneck_scale), w = (int)floor((double)W * (double)bottleneck_scale);
  UD_REQUIRE(h >= 1 && w >= 1, UD_ERR_INVALID, "downscale: %dx%d scaled by %g is empty", H, W, bottleneck_scale);
  const long long total = (long long)planes * H * W;
  if (total == 0) return UD_OK;
  UD_REQUIRE(x && y, UD_ERR_INVALID, "downscale: null pointer");
  // first resize was called with scale_factor -> scale = (float)(1.0 / scale_factor); second with size -> in/out
  const float sd = (float)(1.0 / (double)bottleneck_scale);
  const float suy = (float)h / (float)H, sux = (float)w / (float)W;
  const int blocks = (int)min((long long)UD_NUM_SMS * 8, (total + 255) / 256);
  pt_downscale_kernel<<<blocks, 256, 0, stream>>>(x, y, total, H, W, h, w, sd, sd, suy, sux);
  return ud_check_launch("downscale");
}

// Adjoint of downscale: gx[R,Q] = sum of gy[r,c] over the output pixels whose composite nearest index is (R,Q).  The
// composite index f(r) = min(floor(min(floor(r*suy), h-1) * sdy), H-1) is non-decreasing in r, so the preimage of R is
// the contiguous range [first[R], first[R+1]); each CTA builds first[] for both axes in shared memory with the
// forward's fp32 arithmetic, then every input pixel sums its rectangle in row-major order.
__device__ __forceinline__ int pt_ds_src(int r, int H, int h, float sd, float su) {
  const int rm = min((int)floorf((float)r * su), h - 1);
  return min((int)floorf((float)rm * sd), H - 1);
}

__global__ void __launch_bounds__(256)
pt_downscale_bwd_kernel(const float* __restrict__ gy, float* __restrict__ gx, int H, int W, int h, int w, float sdy,
                        float sdx, float suy, float sux) {
  extern __shared__ int pt_first[];    // rows [H+1] | cols [W+1]
  int* fr = pt_first;
  int* fc = pt_first + H + 1;
  for (int i = threadIdx.x; i <= H; i += blockDim.x) fr[i] = H;
  for (int i = threadIdx.x; i <= W; i += blockDim.x) fc[i] = W;
  __syncthreads();
  for (int r = threadIdx.x; r < H; r += blockDim.x) {   // r is the first preimage row of every R in (f(r-1), f(r)]
    const int f = pt_ds_src(r, H, h, sdy, suy), lo = r ? pt_ds_src(r - 1, H, h, sdy, suy) + 1 : 0;
    for (int R = lo; R <= f; ++R) fr[R] = r;
  }
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    const int f = pt_ds_src(c, W, w, sdx, sux), lo = c ? pt_ds_src(c - 1, W, w, sdx, sux) + 1 : 0;
    for (int Q = lo; Q <= f; ++Q) fc[Q] = c;
  }
  __syncthreads();
  const float* p = gy + (long long)blockIdx.y * H * W;
  float* q = gx + (long long)blockIdx.y * H * W;
  const long long total = (long long)H * W;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int R = (int)(i / W), Q = (int)(i - (long long)R * W);
    float acc = 0.f;
    for (int r = fr[R]; r < fr[R + 1]; ++r)
      for (int c = fc[Q]; c < fc[Q + 1]; ++c) acc += __ldg(p + (long long)r * W + c);
    q[i] = acc;
  }
}

extern "C" int ud_downscale_nearest_bwd(const float* gy, float* gx, int planes, int H, int W, float bottleneck_scale,
                                        cudaStream_t stream) {
  UD_REQUIRE(planes >= 0 && H >= 1 && W >= 1 && bottleneck_scale > 0.f, UD_ERR_INVALID, "downscale_bwd: bad arguments");
  const int h = (int)floor((double)H * (double)bottleneck_scale), w = (int)floor((double)W * (double)bottleneck_scale);
  UD_REQUIRE(h >= 1 && w >= 1, UD_ERR_INVALID, "downscale_bwd: %dx%d scaled by %g is empty", H, W, bottleneck_scale);
  if ((long long)planes * H * W == 0) return UD_OK;
  UD_REQUIRE(gy && gx, UD_ERR_INVALID, "downscale_bwd: null pointer");
  UD_REQUIRE(planes <= 65535, UD_ERR_UNSUPPORTED, "downscale_bwd: too many planes (%d)", planes);
  const size_t smem = sizeof(int) * ((size_t)H + W + 2);
  UD_REQUIRE(smem <= (48u << 10), UD_ERR_UNSUPPORTED, "downscale_bwd: %dx%d planes are too large", H, W);
  const float sd = (float)(1.0 / (double)bottleneck_scale);
  const float suy = (float)h / (float)H, sux = (float)w / (float)W;
  const int per_plane = ud_cdiv((long long)H * W, 256 * 8);     // 8 pixels per thread
  pt_downscale_bwd_kernel<<<dim3(per_plane, planes), 256, smem, stream>>>(gy, gx, H, W, h, w, sd, sd, suy, sux);
  return ud_check_launch("downscale_bwd");
}
