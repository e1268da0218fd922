// Counter-based normals shared by the random corruptions (ud_corrupt.cu) and SmoothGrad (ud_explain.cu); restated
// in numpy by oracle/corrupt.py.
#pragma once

// Philox4x32-10 (Salmon et al., SC'11), as Random123 defines it
__device__ __forceinline__ uint4 ud_philox(uint4 c, unsigned k0, unsigned k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// Box-Muller: u1 = (a + 0.5)*2^-32, u2 = b*2^-32.  ln(u1) goes through log1p(-(1 - u1)) in the upper half, where
// 1 - u1 = (~a + 0.5)*2^-32 is exact in the integer and u1 itself would lose it to fp32 rounding.
__device__ __forceinline__ float2 ud_box_muller(unsigned a, unsigned b) {
  const float l = a < 0x80000000u ? logf(__fmul_rn(__fadd_rn((float)a, 0.5f), 0x1p-32f))
                                  : log1pf(-__fmul_rn(__fadd_rn((float)(~a), 0.5f), 0x1p-32f));
  const float r = sqrtf(-2.f * l);
  float sn, cs;
  sincospif(__fmul_rn((float)b, 0x1p-31f), &sn, &cs);
  return make_float2(r * cs, r * sn);
}
