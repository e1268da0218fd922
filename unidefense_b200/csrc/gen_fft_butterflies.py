#!/usr/bin/env python3
"""Generates ud_fft_bfly_gen.cuh: fully unrolled odd-prime DFT butterflies with literal
twiddle constants (so ptxas emits FFMA with immediate operands).

For prime p, h=(p-1)/2, inputs v[0..p-1] (complex), forward DFT X[k] = sum_j v[j] e^{-2 pi i jk/p}:
    a_q = v[q] + v[p-q],  b_q = v[q] - v[p-q]                       q = 1..h
    X[0]   = v0 + sum_q a_q
    C_k    = v0 + sum_q cos(2 pi qk/p) a_q          (complex)
    S_k    =      sum_q sin(2 pi qk/p) b_q          (complex)
    X[k]   = C_k - i S_k = (C.re + S.im, C.im - S.re)
    X[p-k] = C_k + i S_k = (C.re - S.im, C.im + S.re)
4 h^2 FMAs instead of the 4 p^2 of the plain O(p^2) DFT.

    python gen_fft_butterflies.py > ud_fft_bfly_gen.cuh
"""
import math
import sys

PRIMES = [3, 5, 7, 11, 13, 17, 19, 23]


def lit(x: float) -> str:
    return f"{x:.9e}f"


def gen(p: int) -> str:
    h = (p - 1) // 2
    o = []
    o.append(f"// radix-{p} butterfly, in place, forward sign (e^{{-i}}); {4 * h * h} FMAs")
    o.append(f"__device__ __forceinline__ void ud_bfly{p}(float2 (&v)[{p}]) {{")
    for q in range(1, h + 1):
        o.append(f"  const float ar{q} = v[{q}].x + v[{p - q}].x, ai{q} = v[{q}].y + v[{p - q}].y;")
        o.append(f"  const float br{q} = v[{q}].x - v[{p - q}].x, bi{q} = v[{q}].y - v[{p - q}].y;")
    o.append("  const float v0r = v[0].x, v0i = v[0].y;")
    sr = " + ".join(f"ar{q}" for q in range(1, h + 1))
    si = " + ".join(f"ai{q}" for q in range(1, h + 1))
    o.append(f"  v[0].x = v0r + ({sr});")
    o.append(f"  v[0].y = v0i + ({si});")
    for k in range(1, h + 1):
        o.append("  {")
        o.append("    float cr = v0r, ci = v0i, sr = 0.f, si = 0.f;")
        for q in range(1, h + 1):
            m = (q * k) % p
            c = math.cos(2.0 * math.pi * m / p)
            s = math.sin(2.0 * math.pi * m / p)
            o.append(f"    cr = fmaf({lit(c)}, ar{q}, cr); ci = fmaf({lit(c)}, ai{q}, ci);"
                     f" sr = fmaf({lit(s)}, br{q}, sr); si = fmaf({lit(s)}, bi{q}, si);")
        o.append(f"    v[{k}].x = cr + si; v[{k}].y = ci - sr;")
        o.append(f"    v[{p - k}].x = cr - si; v[{p - k}].y = ci + sr;")
        o.append("  }")
    o.append("}")
    return "\n".join(o)


# Composite radices used by the register-resident two-stage line FFTs (Ud2S, ud_fft.cuh): R = Ra * Rb evaluated as
# Rb sub-DFTs of size Ra, constant twiddles W_R^(nb*ka) (literals), then Ra sub-DFTs of size Rb.  Natural order in
# and out:  v[n], n = Rb*na + nb  ->  X[ka + Ra*kb].
COMPOSITES = [(8, 2, 4), (12, 4, 3), (14, 2, 7), (16, 4, 4), (20, 4, 5)]


def gen_small():
    return """// radix-2 / radix-4 butterflies, forward sign
__device__ __forceinline__ void ud_bfly2(float2 (&v)[2]) {
  const float2 a = v[0], b = v[1];
  v[0] = make_float2(a.x + b.x, a.y + b.y);
  v[1] = make_float2(a.x - b.x, a.y - b.y);
}
__device__ __forceinline__ void ud_bfly4(float2 (&v)[4]) {
  const float s02r = v[0].x + v[2].x, s02i = v[0].y + v[2].y, d02r = v[0].x - v[2].x, d02i = v[0].y - v[2].y;
  const float s13r = v[1].x + v[3].x, s13i = v[1].y + v[3].y, d13r = v[1].x - v[3].x, d13i = v[1].y - v[3].y;
  v[0] = make_float2(s02r + s13r, s02i + s13i);
  v[2] = make_float2(s02r - s13r, s02i - s13i);
  v[1] = make_float2(d02r + d13i, d02i - d13r);
  v[3] = make_float2(d02r - d13i, d02i + d13r);
}"""


def cmul_const(dst: str, src: str, m: int, R: int) -> str:
    """dst = src * exp(-2 pi i m / R) with exact quarter turns."""
    m %= R
    if m == 0:
        return f"{dst} = {src};"
    if 4 * m == R:          # -i
        return f"{dst} = make_float2({src}.y, -{src}.x);"
    if 2 * m == R:          # -1
        return f"{dst} = make_float2(-{src}.x, -{src}.y);"
    if 4 * m == 3 * R:      # +i
        return f"{dst} = make_float2(-{src}.y, {src}.x);"
    c = math.cos(2.0 * math.pi * m / R)
    s = -math.sin(2.0 * math.pi * m / R)
    return (f"{dst} = make_float2(fmaf({lit(c)}, {src}.x, {lit(-s)} * {src}.y), "
            f"fmaf({lit(c)}, {src}.y, {lit(s)} * {src}.x));")


def gen_composite(R: int, Ra: int, Rb: int) -> str:
    o = [f"// radix-{R} butterfly = {Rb} x radix-{Ra}, literal twiddles, {Ra} x radix-{Rb}; in place, natural order",
         f"__device__ __forceinline__ void ud_bfly{R}(float2 (&v)[{R}]) {{", f"  float2 t[{Rb}][{Ra}];"]
    for nb in range(Rb):
        o.append("  {")
        o.append(f"    float2 a[{Ra}] = {{" + ", ".join(f"v[{Rb * na + nb}]" for na in range(Ra)) + "};")
        o.append(f"    ud_bfly{Ra}(a);")
        for ka in range(Ra):
            o.append("    " + cmul_const(f"t[{nb}][{ka}]", f"a[{ka}]", nb * ka, R))
        o.append("  }")
    for ka in range(Ra):
        o.append("  {")
        o.append(f"    float2 b[{Rb}] = {{" + ", ".join(f"t[{nb}][{ka}]" for nb in range(Rb)) + "};")
        o.append(f"    ud_bfly{Rb}(b);")
        for kb in range(Rb):
            o.append(f"    v[{ka + Ra * kb}] = b[{kb}];")
        o.append("  }")
    o.append("}")
    return "\n".join(o)


def main():
    print("// GENERATED by gen_fft_butterflies.py -- do not edit by hand.")
    print("#pragma once")
    print("#ifndef UD_BFLY_HOST_TEST")
    print("#include <cuda_runtime.h>")
    print("#endif")
    print()
    print(gen_small())
    print()
    for p in PRIMES:
        print(gen(p))
        print()
    for R, Ra, Rb in COMPOSITES:
        print(gen_composite(R, Ra, Rb))
        print()


if __name__ == "__main__":
    main()
