// devmath.cuh — device arithmetic that must reproduce the reference's pinned int8 build bit for bit.
// Every float op is an explicit round-to-nearest intrinsic (never contracted); __fmaf_rn appears exactly
// where the reference has _mm256_fmadd_ps.  Citations are to /root/reference/src.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lpcnet_b200 {

#define LPCNET_SCALE   (128.f * 127.f)          // vec_avx.h:686
#define LPCNET_SCALE_1 (1.f / 128.f / 127.f)    // vec_avx.h:687

// _mm256_rcp_ps emulation (vec_avx.h:406,435): Intel RCPPS is a 2048-entry table on the top 11 mantissa bits with
// the exponent negated separately (verified exhaustively by oracle/capture_rcp.py).  tab16[k] = (T[k]-0x3f000000)>>11.
__device__ __forceinline__ float rcp_emul(float x, const uint16_t *__restrict__ tab16)
{
    uint32_t u = __float_as_uint(x);
    uint32_t t = 0x3f000000u + ((uint32_t)tab16[(u >> 12) & 0x7FFu] << 11);
    return __uint_as_float(t - ((u & 0x7F800000u) - 0x3F800000u));
}
// same with the shared-memory table of the per-sample kernel: tab32[k] = T[k] + 0x3f800000 (no re-assembly needed)
__device__ __forceinline__ float rcp_emul(float x, const uint32_t *__restrict__ tab32)
{
    const uint32_t u = __float_as_uint(x);
    // byte offset of entry (u >> 12) & 0x7FF, formed with one shift + one mask
    const uint32_t t = *reinterpret_cast<const uint32_t *>(reinterpret_cast<const char *>(tab32) + ((u >> 10) & 0x1FFCu));
    return __uint_as_float(t - (u & 0x7F800000u));
}

// same table at an 8 KB-aligned SHARED address: the entry address is formed with one shift and one (a & b) | c
struct RcpShared { uint32_t addr; };
__device__ __forceinline__ float rcp_emul(float x, RcpShared tab)
{
    const uint32_t u = __float_as_uint(x);
    uint32_t t;
    asm("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(tab.addr | ((u >> 10) & 0x1FFCu)));
    return __uint_as_float(t - (u & 0x7F800000u));
}

// The same function WITHOUT a table (no shared-memory traffic: the look-up above costs ~3.4 bank-conflicted wavefronts
// per warp, the binding unit of the per-sample kernel).  The table has the closed form T[k] = rint(2^25/d) * 2^-13 with
// d = 2k + 4097 (tests/test_oracle.py): d is formed exactly as a float from the top 11 mantissa bits, MUFU.RCP gives
// 2^25/d to within +-1 after rounding, and the EXACT residual q*d - 2^25 (an integer below 2^24, so one FMA computes
// it without error) decides the +-1 correction; d is odd, so there are no ties.  Checked against the table for every
// k, exponent and sign of the low bits by tests/test_gpu_parity.py::test_arithmetic_rcpps_matches_table.
struct RcpArith {};
__device__ __forceinline__ float rcp_emul(float x, RcpArith)
{
    const uint32_t u = __float_as_uint(x);
    const float d = __uint_as_float((u & 0x007FF000u) | 0x45800800u);        // 4097 + 2k, exact
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(d));
    float q = __fsub_rn(__fmaf_rn(y, 33554432.f, 12582912.f), 12582912.f);   // rint(y * 2^25)
    const float e = __fmaf_rn(q, d, -33554432.f);                           // q*d - 2^25, exact
    const float dh = __fmul_rn(d, 0.5f);
    q = __fadd_rn(__fsub_rn(q, e > dh ? 1.f : 0.f), e < -dh ? 1.f : 0.f);
    // T[k] + 0x3f800000 - exponent(x):  q in [4097, 8191] is 0x45800000 + ((q - 4096) << 11) as a float pattern
    return __uint_as_float(__float_as_uint(q) + 0x39000000u - (u & 0x7F800000u));
}

// tanh8_approx (vec_avx.h:393-411)
template <typename TAB>
__device__ __forceinline__ float tanh_approx(float x, TAB tab16)
{
    const float N0 = 952.52801514f, N1 = 96.39235687f, N2 = 0.60863042f;
    const float D0 = 952.72399902f, D1 = 413.36801147f, D2 = 11.88600922f;
    float X2 = __fmul_rn(x, x);
    float num = __fmaf_rn(__fmaf_rn(N2, X2, N1), X2, N0);
    float den = __fmaf_rn(__fmaf_rn(D2, X2, D1), X2, D0);
    num = __fmul_rn(num, x);
    den = rcp_emul(den, tab16);
    num = __fmul_rn(num, den);
    return fmaxf(-1.f, fminf(1.f, num));
}

// sigmoid8_approx (vec_avx.h:421-440)
template <typename TAB>
__device__ __forceinline__ float sigmoid_approx(float x, TAB tab16)
{
    const float N0 = 238.13200378f, N1 = 6.02452230f, N2 = 0.00950985f;
    const float D0 = 952.72399902f, D1 = 103.34200287f, D2 = 0.74287558f;
    float X2 = __fmul_rn(x, x);
    float num = __fmaf_rn(__fmaf_rn(N2, X2, N1), X2, N0);
    float den = __fmaf_rn(__fmaf_rn(D2, X2, D1), X2, D0);
    num = __fmul_rn(num, x);
    den = rcp_emul(den, tab16);
    num = __fmaf_rn(num, den, 0.5f);
    return fmaxf(0.f, fminf(1.f, num));
}

// ---- Blackwell packed fp32 (two lanes per 64-bit register pair: FFMA2 / FMUL2 / FADD2) ----
// Used for the pieces of the activations where both neurons of a lane run the same op.  ptxas contracts a packed
// multiply followed by a packed add into one FFMA2 even with -fmad=false (observed), which would change the rounding,
// so the packed forms are applied ONLY where the reference has an fma, a lone multiply, or an add whose result is
// multiplied (add -> mul cannot be contracted); every mul -> add of the reference stays scalar.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 k2(float c) { return pk2(c, c); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// 1 - z for two values: fma(z, -1, 1) = rn(1 - z)
__device__ __forceinline__ f32x2 one_minus2(f32x2 z) { return fma2(z, k2(-1.f), k2(1.f)); }
// x + y where x (and maybe y) is the result of a packed multiply: written as fma(x, ONE, y) = rn(x*1 + y) = rn(x + y) with a ONE = {1.f, 1.f}
// that the compiler cannot see through (it is read from shared memory at kernel start), so the multiply that produced x cannot be
// contracted into it — which ptxas does to a packed mul followed by a packed add (see above).  Same instruction count as an add.
__device__ __forceinline__ f32x2 oadd2(f32x2 x, f32x2 one, f32x2 y) { return fma2(x, one, y); }
// numerator * x and denominator of the rational approximations (before the reciprocal), two values at a time:
// X2 = x*x; num = fma(fma(N2,X2,N1),X2,N0) * x; den = fma(fma(D2,X2,D1),X2,D0)          (vec_avx.h:393-440)
__device__ __forceinline__ void rational2(f32x2 x, float N0, float N1, float N2, float D0, float D1, float D2, f32x2 &num, f32x2 &den)
{
    const f32x2 X2 = mul2(x, x);
    num = fma2(fma2(k2(N2), X2, k2(N1)), X2, k2(N0));
    den = fma2(fma2(k2(D2), X2, k2(D1)), X2, k2(D0));
    num = mul2(num, x);
}
#define LPCNET_SIGMOID_COEF 238.13200378f, 6.02452230f, 0.00950985f, 952.72399902f, 103.34200287f, 0.74287558f
#define LPCNET_TANH_COEF 952.52801514f, 96.39235687f, 0.60863042f, 952.72399902f, 413.36801147f, 11.88600922f
// (float)acc * SCALE_1 for two biased accumulators (see acc_init_t below): add -> mul, safe to pack
__device__ __forceinline__ f32x2 acc_finish2(int a0, int a1)
{
    return mul2(add2(pk2(__int_as_float(a0), __int_as_float(a1)), k2(-12582912.f)), k2(LPCNET_SCALE_1));
}

// vector_ps_to_epi8 (vec_avx.h:321-336): u8 = sat(rne(fma(x,127,127)))
__device__ __forceinline__ uint32_t quant_u8(float x)
{
    int v = __float2int_rn(__fmaf_rn(x, 127.f, 127.f));
    return (uint32_t)min(255, max(0, v));
}

// accumulator entry/exit of the int8 GEMVs (vec_avx.h:803-806,854-856)
__device__ __forceinline__ int acc_init(float rec) { return __float2int_rn(__fmul_rn(rec, LPCNET_SCALE)); }
__device__ __forceinline__ float acc_finish(int acc) { return __fmul_rn(__int2float_rn(acc), LPCNET_SCALE_1); }

// The same two conversions without the conversion unit, for models whose pre-activations are PROVEN (model.cu,
// cvt_range_ok) to stay below 2^22 in accumulator units: adding 1.5*2^23 to |v| < 2^22 rounds v to the nearest-even
// integer exactly like cvtps2dq and leaves 0x4B400000 + rne(v) in the float's bit pattern; the accumulator keeps that
// bias while the integer GEMV sum is added, and subtracting 1.5*2^23 from the biased pattern is exactly (float)acc.
#define LPCNET_CVT_MAGIC 12582912.f              // 1.5 * 2^23 = 0x4B400000
template <bool FAST> __device__ __forceinline__ int acc_init_t(float rec)
{
    if (FAST) return __float_as_int(__fadd_rn(__fmul_rn(rec, LPCNET_SCALE), LPCNET_CVT_MAGIC));
    return acc_init(rec);
}
template <bool FAST> __device__ __forceinline__ float acc_finish_t(int acc)
{
    if (FAST) return __fmul_rn(__fsub_rn(__int_as_float(acc), LPCNET_CVT_MAGIC), LPCNET_SCALE_1);
    return acc_finish(acc);
}
// quantised byte of a state value |h| <= 1 (fma(h,127,127) in [0,254]: the saturation of vector_ps_to_epi8 cannot trigger);
// FAST leaves it in the low byte of the biased pattern
template <bool FAST> __device__ __forceinline__ uint32_t quant_u8_t(float x)
{
    if (FAST) return __float_as_uint(__fadd_rn(__fmaf_rn(x, 127.f, 127.f), LPCNET_CVT_MAGIC));
    return quant_u8(x);
}

// u8 activations x s8 weights, 4 MACs (one block row of sparse_sgemv_accum8x4; maddubs+madd == exact integer sum
// under the WeightClip pair constraint, training_tf2/lpcnet.py:216-232)
__device__ __forceinline__ int dp4a_us(uint32_t x_u8x4, int w_s8x4, int acc)
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(x_u8x4), "r"(w_s8x4), "r"(acc));
    return d;
}

// log2_approx + lin2ulaw (common.h:18-33,47-58)
__device__ __forceinline__ float log2_approx(float x)
{
    int i = __float_as_int(x);
    int integer = (i >> 23) - 127;
    i -= integer << 23;
    float frac = __fsub_rn(__int_as_float(i), 1.5f);
    frac = __fadd_rn(-0.41445418f, __fmul_rn(frac, __fadd_rn(0.95909232f,
           __fmul_rn(frac, __fadd_rn(-0.33951290f, __fmul_rn(frac, 0.16541097f))))));
    return __fadd_rn(__int2float_rn(1 + integer), frac);
}
__device__ __forceinline__ int lin2ulaw(float x)
{
    const float scale = 255.f / 32768.f;
    float s = x >= 0 ? 1.f : -1.f;
    x = fabsf(x);
    float l = __fmul_rn(0.69315f, log2_approx(__fadd_rn(1.f, __fmul_rn(scale, x))));
    float u = __fmul_rn(s, __fdiv_rn(__fmul_rn(128.f, l), 5.5451774445f));
    u = __fadd_rn(128.f, u);
    if (u < 0) u = 0;
    if (u > 255) u = 255;
    return __double2int_rd(0.5 + (double)u);     // (int)floor(.5 + u), evaluated in double like the reference
}

// kiss99_rand (kiss99.c:59-81)
struct Kiss99 { uint32_t z, w, jsr, jcong; };
__device__ __forceinline__ uint32_t kiss99_rand(Kiss99 &t)
{
    uint32_t znew = 36969u * (t.z & 0xFFFFu) + (t.z >> 16);
    uint32_t wnew = 18000u * (t.w & 0xFFFFu) + (t.w >> 16);
    uint32_t mwc = (znew << 16) + wnew;
    uint32_t shr3 = t.jsr ^ (t.jsr << 13);
    shr3 ^= shr3 >> 17;
    shr3 ^= shr3 << 5;
    uint32_t cong = 69069u * t.jcong + 1234567u;
    t.z = znew; t.w = wnew; t.jsr = shr3; t.jcong = cong;
    return (mwc ^ cong) + shr3;
}

__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

}  // namespace lpcnet_b200
