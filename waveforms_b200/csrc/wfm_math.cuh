// wfm_math.cuh — correctly-rounded, never-contracted fp64 primitives.
// NumPy / SciPy evaluate a*b+c as two rounded operations; these wrappers keep
// the compiler from fusing them (see wfm_basis.cuh, wfm_iir.cu).
#pragma once
#include <stdint.h>

namespace wfm {

__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dvd(double a, double b) { return __ddiv_rn(a, b); }

// sin and cos of one argument with a Cody-Waite reduction that stays on the fast
// path up to |a| = 2^30 (CUDA's sincos() leaves it at 105615 rad and then calls a
// Payne-Hanek routine with a local-memory scratch array: a 200 MHz carrier passes
// that threshold 84 us into a frame).  pi/2 = HI + MID + LO (round-to-nearest
// splits); q*HI is subtracted exactly by the first FMA (the difference is a
// multiple of 2^-52 below 2), the next two carry the tail, so the reduced
// argument has a relative error of ~2^-53 even next to a multiple of pi/2.
// Kernels: the fdlibm minimax polynomials on [-pi/4, pi/4].  Measured against
// mpmath over +-1e9 (incl. neighbours of k*pi/2): relative error < 2 * 2^-53.
// The coefficients sit in constant memory so that every FMA takes its constant
// as a c[bank][offset] operand instead of two moves into registers.
static __constant__ double kTrig[16] = {
    0.6366197723675814,        // 0: 2/pi
    1.5707963267948966,        // 1: pi/2 HI
    6.123233995736766e-17,     // 2: pi/2 MID
    -1.4973849048591698e-33,   // 3: pi/2 LO
    1.58969099521155010221e-10,   // 4: S6
    -2.50507602534068634195e-08,  // 5: S5
    2.75573137070700676789e-06,   // 6: S4
    -1.98412698298579493134e-04,  // 7: S3
    8.33333333332248946124e-03,   // 8: S2
    -1.66666666666666324348e-01,  // 9: S1
    -1.13596475577881948265e-11,  // 10: C6
    2.08757232129817482790e-09,   // 11: C5
    -2.75573143513906633035e-07,  // 12: C4
    2.48015872894767294178e-05,   // 13: C3
    -1.38888888888741095749e-03,  // 14: C2
    4.16666666666666019037e-02,   // 15: C1
};

struct SinCos {
  double s, c;
};

static __device__ __noinline__ SinCos sincos_huge(double a) {  // CUDA's Payne-Hanek path, out of line
  SinCos r;
  sincos(a, &r.s, &r.c);
  return r;
}

__device__ __forceinline__ SinCos sincos_cw(double a) {
  if (!(fabs(a) <= 1073741824.0)) return sincos_huge(a);  // also NaN / inf
  const double q = rint(a * kTrig[0]);
  double r = fma(-q, kTrig[1], a);
  r = fma(-q, kTrig[2], r);
  r = fma(-q, kTrig[3], r);
  const double z = r * r;
  double ps = kTrig[4];
  ps = fma(ps, z, kTrig[5]);
  ps = fma(ps, z, kTrig[6]);
  ps = fma(ps, z, kTrig[7]);
  ps = fma(ps, z, kTrig[8]);
  ps = fma(ps, z, kTrig[9]);
  const double s = fma(r * z, ps, r);
  double pc = kTrig[10];
  pc = fma(pc, z, kTrig[11]);
  pc = fma(pc, z, kTrig[12]);
  pc = fma(pc, z, kTrig[13]);
  pc = fma(pc, z, kTrig[14]);
  pc = fma(pc, z, kTrig[15]);
  const double hz = 0.5 * z;
  const double w = 1.0 - hz;
  const double c = w + (((1.0 - w) - hz) + z * z * pc);
  const int n = (int)q;
  // quadrant: swap for odd n, then flip signs through the sign bit
  const bool odd = n & 1;
  const double ss = odd ? c : s;
  const double cc = odd ? s : c;
  const unsigned long long sbit = (unsigned long long)(n & 2) << 62;
  const unsigned long long cbit = (unsigned long long)((n + 1) & 2) << 62;
  SinCos o;
  o.s = __longlong_as_double(__double_as_longlong(ss) ^ sbit);
  o.c = __longlong_as_double(__double_as_longlong(cc) ^ cbit);
  return o;
}

__device__ __forceinline__ double sin_cw(double a) { return sincos_cw(a).s; }
__device__ __forceinline__ double cos_cw(double a) { return sincos_cw(a).c; }

// N independent arguments at once: the same arithmetic per element (bit-identical to
// sincos_cw), written element-wise so that the N dependency chains interleave.
template <int N>
__device__ __forceinline__ void sincos_cw_n(const double (&a)[N], double (&s_out)[N], double (&c_out)[N]) {
  bool fast = true;
#pragma unroll
  for (int u = 0; u < N; ++u) fast = fast && (fabs(a[u]) <= 1073741824.0);
  if (!fast) {
#pragma unroll
    for (int u = 0; u < N; ++u) {
      const SinCos r = sincos_cw(a[u]);
      s_out[u] = r.s;
      c_out[u] = r.c;
    }
    return;
  }
  double q[N], r[N], z[N], ps[N], pc[N];
#pragma unroll
  for (int u = 0; u < N; ++u) q[u] = rint(a[u] * kTrig[0]);
#pragma unroll
  for (int u = 0; u < N; ++u) r[u] = fma(-q[u], kTrig[1], a[u]);
#pragma unroll
  for (int u = 0; u < N; ++u) r[u] = fma(-q[u], kTrig[2], r[u]);
#pragma unroll
  for (int u = 0; u < N; ++u) r[u] = fma(-q[u], kTrig[3], r[u]);
#pragma unroll
  for (int u = 0; u < N; ++u) {
    z[u] = r[u] * r[u];
    ps[u] = kTrig[4];
    pc[u] = kTrig[10];
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) {
#pragma unroll
    for (int u = 0; u < N; ++u) {
      ps[u] = fma(ps[u], z[u], kTrig[5 + k]);
      pc[u] = fma(pc[u], z[u], kTrig[11 + k]);
    }
  }
#pragma unroll
  for (int u = 0; u < N; ++u) {
    const double s = fma(r[u] * z[u], ps[u], r[u]);
    const double hz = 0.5 * z[u];
    const double w = 1.0 - hz;
    const double c = w + (((1.0 - w) - hz) + z[u] * z[u] * pc[u]);
    const int n = (int)q[u];
    const bool odd = n & 1;
    const double ss = odd ? c : s;
    const double cc = odd ? s : c;
    const unsigned long long sbit = (unsigned long long)(n & 2) << 62;
    const unsigned long long cbit = (unsigned long long)((n + 1) & 2) << 62;
    s_out[u] = __longlong_as_double(__double_as_longlong(ss) ^ sbit);
    c_out[u] = __longlong_as_double(__double_as_longlong(cc) ^ cbit);
  }
}

// The 16-bit DAC code of a sample v on a row with gain g and offset o (WFM_I16 output, wfm_quantize):
//   clamp(rint(v * g + o), -32768, 32767)   multiply, then add (never fused); rint rounds half to even
// NaN -> 0 (tested here, not left to the conversion instruction); +-inf saturate like any out-of-range value.
// The clamp runs on the integer: cvt.rni.s32.f64 saturates at the int32 range (PTX: float-to-integer conversions
// clamp to the destination range), and the two fp64 min / max it saves are issue slots of the FP64 pipe, which the
// dense kernel is bound by.
__device__ __forceinline__ int16_t dac_code(double v, double g, double o) {
  const double y = add(mul(v, g), o);
  if (y != y) return 0;
  return (int16_t)min(max(__double2int_rn(y), -32768), 32767);
}

}  // namespace wfm
