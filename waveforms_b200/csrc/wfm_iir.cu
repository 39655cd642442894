// wfm_iir.cu — K2: IIR filters with the semantics of scipy.signal.sosfilt and scipy.signal.lfilter.
//
// Replaces the sosfilt call sites of the reference's waveforms/waveform.py:200-203 and :249 and the lfilter of its
// waveforms/distortion.py:321.  Per biquad section, direct form II transposed, exactly the recurrence scipy runs
// (scipy/signal/_sosfilt.pyx):
//     y  = b0*x + z0
//     z0 = b1*x - a1*y + z1
//     z1 = b2*x - a2*y
// and for lfilter scipy's direct-form loop (lfilter_step below), with every product and sum rounded separately
// (no FMA; built with -fmad=false and written with __dmul_rn/__dadd_rn).
//
// Three kernels:
//
//  * sosfilt_exact_kernel, lfilter_exact_kernel (WFM_IIR_EXACT) — one warp per signal walks time sequentially with
//    scipy's recurrence.  Bit-identical to scipy.
//
//  * iir_scan_kernel<Form, kAligned> (WFM_IIR_SCAN) — block-parallel associative scan, shared by both filters.  Each
//    is a linear system on its D state words, s' = M s + g x: a cascade of one or two biquads on the joint state of
//    its sections (BiquadForm, D = 2 S; longer cascades run as a chain of launches) or lfilter's direct form of
//    order 1..4 (DirectForm, D = M).  One CTA per signal walks 4096-sample tiles; inside a tile each of 256 threads
//    owns 16 consecutive samples:
//       pass a: every thread runs its chunk from the zero state in state-space form (one FMA per step on the
//               critical path) -> its end state f_i (thread 0 starts from the tile's carry-in state);
//       scan  : E_i = sum_{j<i} (M^16)^(i-1-j) f_j  (warp shuffles, then 8 warp totals through shared memory; the
//               D x D powers of M^16 come from the host, computed in long double);
//       pass c: every thread re-runs its chunk from E_i with scipy's own recurrence and writes y.
//    The result differs from the sequential one only through the rounding of the carried states: ~1e-16 * (filter
//    noise gain).  For poles within 5e-3 of the unit circle (the exp-decay predistortion filters) that noise gain
//    makes scipy's OWN sequential result uncertain at the 3e-12 level, which no re-association can track
//    (DESIGN.md §K2); for well-conditioned filters the two modes agree to ~1e-15.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstring>
#include "wfm_internal.h"
#include "wfm_math.cuh"

namespace wfm {

constexpr int kIirThreads = 256;
constexpr int kIirT = 16;                          // samples per thread per tile
constexpr int kIirTile = kIirThreads * kIirT;      // 4096
constexpr int kIirMinBlocks = 2;                   // CTAs per SM the scan kernel is compiled for
constexpr int kMaxSections = 8;

struct Biquad {
  double b0, b1, b2, a1, a2;
};

struct IirParams {
  int n_sections;
  int shift_in, shift_out;  // scan only: subtract `initial` at the input / add it at the output of THIS launch
  double initial;
  Biquad sec[kMaxSections];
};

__device__ __forceinline__ void biquad_step(const Biquad& q, double x, double& z0, double& z1, double& y) {
  y = add(mul(q.b0, x), z0);
  z0 = add(sub(mul(q.b1, x), mul(q.a1, y)), z1);
  z1 = sub(mul(q.b2, x), mul(q.a2, y));
}

// ---------------------------------------------------------------------------
// exact: ONE WARP per signal, sequential in time.  The warp loads 32 consecutive
// samples with one coalesced access (the next block is already in flight), every lane
// runs the same recurrence on the broadcast samples (the state is replicated, so no
// lane waits for another) and lane l keeps output l: loads and stores are full lines
// and the only serial cost left is the recurrence's own dependency chain.
// ---------------------------------------------------------------------------
constexpr int kExactWarps = 4;  // warps (= signals) per CTA

__device__ __forceinline__ double shfl_f64(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

__global__ void __launch_bounds__(32 * kExactWarps) sosfilt_exact_kernel(const __grid_constant__ IirParams P,
                                                                         const double* __restrict__ x, double* y,
                                                                         int64_t n_sig, int64_t n, int64_t stride,
                                                                         const double* __restrict__ zi,
                                                                         double* __restrict__ zf) {
  const int lane = threadIdx.x & 31;
  const int64_t s = (int64_t)blockIdx.x * kExactWarps + (threadIdx.x >> 5);
  if (s >= n_sig) return;
  const int S = P.n_sections;
  double z0[kMaxSections], z1[kMaxSections];
#pragma unroll
  for (int k = 0; k < kMaxSections; ++k) {
    z0[k] = (zi && k < S) ? zi[(s * S + k) * 2 + 0] : 0.0;
    z1[k] = (zi && k < S) ? zi[(s * S + k) * 2 + 1] : 0.0;
  }
  const double* __restrict__ xs = x + s * stride;
  double* ys = y + s * stride;
  const bool shift = P.initial != 0.0;
  double nxt = lane < n ? xs[lane] : 0.0;
  for (int64_t base = 0; base < n; base += 32) {
    const double mine = nxt;
    if (base + 32 + lane < n) nxt = xs[base + 32 + lane];  // in flight while this block is filtered
    const int cnt = (int)min((int64_t)32, n - base);
    double out = 0.0;
    if (S == 1 && cnt == 32) {  // full blocks of the common cases: no branch between the samples, so the
      const Biquad q = P.sec[0];  // 32 broadcasts are issued ahead of the recurrence that consumes them
#pragma unroll
      for (int l = 0; l < 32; ++l) {
        double cur = shfl_f64(mine, l), o;
        if (shift) cur = sub(cur, P.initial);
        biquad_step(q, cur, z0[0], z1[0], o);
        if (lane == l) out = o;
      }
    } else if (S == 2 && cnt == 32) {
      // software-pipelined across the sections: section 1 of sample l next to section 2 of sample l - 1 — two
      // independent dependency chains in flight, the same operations in the same order per section (bit-identical)
      const Biquad q0 = P.sec[0], q1 = P.sec[1];
      double o1_prev;
      {
        double cur = shfl_f64(mine, 0);
        if (shift) cur = sub(cur, P.initial);
        biquad_step(q0, cur, z0[0], z1[0], o1_prev);
      }
#pragma unroll
      for (int l = 1; l <= 32; ++l) {
        double o1 = 0.0, o2;
        if (l < 32) {
          double cur = shfl_f64(mine, l);
          if (shift) cur = sub(cur, P.initial);
          biquad_step(q0, cur, z0[0], z1[0], o1);
        }
        biquad_step(q1, o1_prev, z0[1], z1[1], o2);
        if (lane == l - 1) out = o2;
        o1_prev = o1;
      }
    } else {
#pragma unroll 1
      for (int l = 0; l < cnt; ++l) {
        double cur = shfl_f64(mine, l);
        if (shift) cur = sub(cur, P.initial);
#pragma unroll
        for (int k = 0; k < kMaxSections; ++k)
          if (k < S) {
            double o;
            biquad_step(P.sec[k], cur, z0[k], z1[k], o);
            cur = o;
          }
        if (lane == l) out = cur;
      }
    }
    if (lane < cnt) ys[base + lane] = shift ? add(out, P.initial) : out;
  }
  if (zf && lane == 0) {
#pragma unroll
    for (int k = 0; k < kMaxSections; ++k)
      if (k < S) {
        zf[(s * S + k) * 2 + 0] = z0[k];
        zf[(s * S + k) * 2 + 1] = z1[k];
      }
  }
}

// ---------------------------------------------------------------------------
// lfilter: single high-order section, scipy.signal.lfilter's DF2T loop
// (scipy/signal/_lfilter.c.src): y = z[0] + b[0]*x;
// z[k] = (z[k+1] + x*b[k+1]) - y*a[k+1];  z[M-1] = x*b[M] - y*a[M].
// Bit-faithful (note the different association from sosfilt's (b1*x - a1*y) + z1).
// ---------------------------------------------------------------------------
constexpr int kMaxOrder = 16;
struct LfilterParams {
  int order;  // M = max(len(a), len(b)) - 1
  double b[kMaxOrder + 1];  // normalised by a[0]
  double a[kMaxOrder + 1];
};

// one lfilter step of order M on the state z[0..M-1] (the exact kernel's replicated state, the scan's chunk state)
template <int M, int N>
__device__ __forceinline__ double lfilter_step(const LfilterParams& P, double xv, double (&z)[N]) {
  if (M == 0) return mul(P.b[0], xv);
  const double yv = add(z[0], mul(P.b[0], xv));
#pragma unroll
  for (int k = 0; k < M - 1; ++k) z[k] = sub(add(z[k + 1], mul(xv, P.b[k + 1])), mul(yv, P.a[k + 1]));
  z[M - 1] = sub(mul(xv, P.b[M]), mul(yv, P.a[M]));
  return yv;
}
__device__ __forceinline__ double lfilter_step_any(const LfilterParams& P, double xv, double (&z)[kMaxOrder]) {
  const int M = P.order;
  if (M == 0) return mul(P.b[0], xv);
  const double yv = add(z[0], mul(P.b[0], xv));
#pragma unroll
  for (int k = 0; k < kMaxOrder - 1; ++k)
    if (k < M - 1) z[k] = sub(add(z[k + 1], mul(xv, P.b[k + 1])), mul(yv, P.a[k + 1]));
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k)
    if (k == M - 1) z[k] = sub(mul(xv, P.b[M]), mul(yv, P.a[M]));
  return yv;
}

// ONE WARP per signal (see sosfilt_exact_kernel): coalesced block loads, the recurrence
// replicated in every lane, lane l keeps output l
__global__ void __launch_bounds__(32 * kExactWarps) lfilter_exact_kernel(const __grid_constant__ LfilterParams P,
                                                                         const double* __restrict__ x, double* y,
                                                                         int64_t n_sig, int64_t n, int64_t stride,
                                                                         const double* __restrict__ zi,
                                                                         double* __restrict__ zf) {
  const int lane = threadIdx.x & 31;
  const int64_t s = (int64_t)blockIdx.x * kExactWarps + (threadIdx.x >> 5);
  if (s >= n_sig) return;
  const int M = P.order;
  double z[kMaxOrder];
#pragma unroll
  for (int k = 0; k < kMaxOrder; ++k) z[k] = (zi && k < M) ? zi[s * M + k] : 0.0;
  const double* __restrict__ xs = x + s * stride;
  double* ys = y + s * stride;
  double nxt = lane < n ? xs[lane] : 0.0;
  for (int64_t base = 0; base < n; base += 32) {
    const double mine = nxt;
    if (base + 32 + lane < n) nxt = xs[base + 32 + lane];
    const int cnt = (int)min((int64_t)32, n - base);
    double out = 0.0;
    if (M == 1 && cnt == 32) {  // full blocks: no branch between the samples (see sosfilt_exact_kernel)
#pragma unroll
      for (int l = 0; l < 32; ++l) {
        const double o = lfilter_step<1>(P, shfl_f64(mine, l), z);
        if (lane == l) out = o;
      }
    } else if (M == 2 && cnt == 32) {
#pragma unroll
      for (int l = 0; l < 32; ++l) {
        const double o = lfilter_step<2>(P, shfl_f64(mine, l), z);
        if (lane == l) out = o;
      }
    } else {
#pragma unroll 1
      for (int l = 0; l < cnt; ++l) {
        const double o = lfilter_step_any(P, shfl_f64(mine, l), z);
        if (lane == l) out = o;
      }
    }
    if (lane < cnt) ys[base + lane] = out;
  }
  if (zf && lane == 0) {
#pragma unroll
    for (int k = 0; k < kMaxOrder; ++k)
      if (k < M) zf[s * M + k] = z[k];
  }
}

// ---------------------------------------------------------------------------
// scan: one CTA per signal, tiles of 4096 samples (see the top of the file)
// ---------------------------------------------------------------------------
constexpr int kMaxJoint = 4;  // largest D: two biquad sections, or lfilter of order 4
struct IirJointTables {
  double lane[32][kMaxJoint * kMaxJoint];  // (M^16)^l, l = 0..31, row-major D x D
  double lvl[5][kMaxJoint * kMaxJoint];    // (M^16)^(2^d)
  double warp[kMaxJoint * kMaxJoint];      // (M^16)^32
  double c[kMaxJoint];                     // state-space input gain of every state word (pass a)
};

template <int D>
__device__ __forceinline__ void matvec_d(const double* __restrict__ M, const double (&a)[D], double (&r)[D]) {
#pragma unroll
  for (int i = 0; i < D; ++i) {
    double acc = M[i * D] * a[0];
#pragma unroll
    for (int j = 1; j < D; ++j) acc = fma(M[i * D + j], a[j], acc);
    r[i] = acc;
  }
}

// What the two filters do differently inside the scan kernel, each a small device-side type:
//   D                          state words per signal;
//   enter(v, valid), leave(v)  the input / output offset of the chunk's samples;
//   state_step(x, f)           pass a: one sample through the state-space form, z' = A z + c x (c in the tables);
//   filter(v, z, ...)          pass c: scipy's recurrence over the chunk from the carried-in state z, in place on v;
//                              where the signal ends inside the chunk (tail_here) `fin` takes the state at sample
//                              `valid`, the final state;
//   state_stride(zs)           state words between two signals in zi / zf: a biquad launch may work on a slice of a
//                              longer cascade's states (zs), a direct form owns all of its D words (a compile-time
//                              stride keeps the order-4 kernel clear of spills);
//   Params                     the kernel parameter block of the coefficients; kMax the largest template argument.

// Cascade of S = 1 or 2 biquads on the joint state (z0, z1) of its sections, D = 2 S.  Section k's state-space step
// is z0' = -a1 z0 + (z1 + c1 u), z1' = -a2 z0 + c2 u (c1 = b1 - a1 b0, c2 = b2 - a2 b0) on its input u, the output of
// section k - 1.  Pass c runs the sections software-pipelined: section 1 of sample k+1 next to section 2 of sample k,
// two independent dependency chains.
template <int S>
struct BiquadForm {
  static constexpr int D = 2 * S, kMax = 2;
  using Params = IirParams;
  __device__ static constexpr int state_stride(int zs) { return zs; }
  Biquad q[S];
  double c1[S], c2[S];
  double initial;
  bool shift_in, shift_out;

  __device__ __forceinline__ BiquadForm(const IirParams& P, const IirJointTables& T)
      : initial(P.initial), shift_in(P.initial != 0.0 && P.shift_in), shift_out(P.initial != 0.0 && P.shift_out) {
#pragma unroll
    for (int k = 0; k < S; ++k) {
      q[k] = P.sec[k];
      c1[k] = T.c[2 * k];
      c2[k] = T.c[2 * k + 1];
    }
  }
  __device__ __forceinline__ void enter(double (&v)[kIirT], int valid) const {
    if (shift_in) {
#pragma unroll
      for (int k = 0; k < kIirT; ++k) v[k] = k < valid ? sub(v[k], initial) : 0.0;
    }
  }
  __device__ __forceinline__ void leave(double (&v)[kIirT]) const {
    if (shift_out) {
#pragma unroll
      for (int k = 0; k < kIirT; ++k) v[k] = add(v[k], initial);
    }
  }
  __device__ __forceinline__ void state_step(double in, double (&f)[D]) const {
#pragma unroll
    for (int sct = 0; sct < S; ++sct) {
      const double z0 = f[2 * sct], z1 = f[2 * sct + 1];
      const double out = fma(q[sct].b0, in, z0);
      f[2 * sct] = fma(-q[sct].a1, z0, fma(c1[sct], in, z1));
      f[2 * sct + 1] = fma(-q[sct].a2, z0, c2[sct] * in);
      in = out;
    }
  }
  __device__ __forceinline__ void filter(double (&v)[kIirT], double (&z)[D], bool tail_here, int valid,
                                         double (&fin)[D]) const {
    if constexpr (S == 1) {
#pragma unroll
      for (int k = 0; k < kIirT; ++k) {
        if (tail_here && k == valid) { fin[0] = z[0]; fin[1] = z[1]; }
        double out;
        biquad_step(q[0], v[k], z[0], z[1], out);
        v[k] = out;
      }
    } else {
      double o1_prev;
      {
        if (tail_here && valid == 0) { fin[0] = z[0]; fin[1] = z[1]; }
        biquad_step(q[0], v[0], z[0], z[1], o1_prev);
      }
#pragma unroll
      for (int k = 1; k <= kIirT; ++k) {
        double o1 = 0.0, o2;
        if (k < kIirT) {
          if (tail_here && k == valid) { fin[0] = z[0]; fin[1] = z[1]; }
          biquad_step(q[0], v[k], z[0], z[1], o1);
        }
        if (tail_here && k - 1 == valid) { fin[2] = z[2]; fin[3] = z[3]; }
        biquad_step(q[1], o1_prev, z[2], z[3], o2);
        v[k - 1] = o2;
        o1_prev = o1;
      }
    }
  }
};

// lfilter's direct form of order M = 1..4, D = M: its DF2T state is z' = A z + c x with A[i][0] = -a[i+1],
// A[i][i+1] = 1 and c[i] = b[i+1] - a[i+1] b[0]; pass c is lfilter_step, the operations of the exact kernel.
template <int M>
struct DirectForm {
  static constexpr int D = M, kMax = 4;
  using Params = LfilterParams;
  __device__ static constexpr int state_stride(int) { return D; }
  const LfilterParams& P;
  const double* c;

  __device__ __forceinline__ DirectForm(const LfilterParams& P_, const IirJointTables& T) : P(P_), c(T.c) {}
  __device__ __forceinline__ void enter(double (&)[kIirT], int) const {}
  __device__ __forceinline__ void leave(double (&)[kIirT]) const {}
  __device__ __forceinline__ void state_step(double in, double (&f)[D]) const {
    const double z0 = f[0];
#pragma unroll
    for (int i = 0; i < D - 1; ++i) f[i] = fma(-P.a[i + 1], z0, fma(c[i], in, f[i + 1]));
    f[D - 1] = fma(-P.a[D], z0, c[D - 1] * in);
  }
  __device__ __forceinline__ void filter(double (&v)[kIirT], double (&z)[D], bool tail_here, int valid,
                                         double (&fin)[D]) const {
#pragma unroll
    for (int k = 0; k < kIirT; ++k) {
      if (tail_here && k == valid) {
#pragma unroll
        for (int i = 0; i < D; ++i) fin[i] = z[i];
      }
      v[k] = lfilter_step<M>(P, v[k], z);
    }
  }
};

// Tile staging: rows of 16 samples at a pitch of 18 doubles (144 B): thread r reads / writes its row with 16-byte
// accesses without bank conflicts, and 16-byte chunks stay aligned for cp.async.  Two buffers: the NEXT tile is
// already on its way (cp.async, no registers held) while this one is filtered — a one-buffer kernel spent three
// quarters of its time waiting for its own loads (ncu: long-scoreboard stalls on the first use of every loaded sample).
constexpr int kJointPitch = kIirT + 2;                                            // doubles per staged row
constexpr int kJointTileBytes = kIirThreads * kJointPitch * (int)sizeof(double);  // 36 864
static_assert(kIirT == 16, "staging puts two-sample chunk c at row c >> 3, column 2 (c & 7): 8 chunks per row");
static_assert(kJointPitch % 2 == 0 && (kJointPitch / 2) % 2 == 1,
              "rows start on 16-byte boundaries at an odd number of 16-byte words apart (no bank conflicts)");
extern __shared__ __align__(16) unsigned char iir_smem[];

__device__ __forceinline__ void cp_async16_zfill(void* dst_smem, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src),
               "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// kAligned: x and y rows start on 16-byte boundaries (cp.async loads, 16-byte stores); else plain 8-byte accesses.
// zi / zf: signal s's state is zi[s * Form::state_stride(zs) + 0 .. D - 1]; a long biquad cascade runs as a chain of
// launches over its sections two by two, each on its slice of the states of the whole cascade (zs = 2 x all its
// sections).
template <class Form, bool kAligned>
__global__ void __launch_bounds__(kIirThreads, kIirMinBlocks) iir_scan_kernel(
    const __grid_constant__ typename Form::Params P, const __grid_constant__ IirJointTables TT, const double* __restrict__ x,
    double* y, int64_t n, int64_t stride, const double* __restrict__ zi, double* __restrict__ zf, int zs) {
  constexpr int D = Form::D;
  double* s_buf0 = reinterpret_cast<double*>(iir_smem);
  double* s_buf1 = reinterpret_cast<double*>(iir_smem + kJointTileBytes);
  __shared__ double s_lane[D * D][32];  // (M^16)^lane, entry-major: conflict-free
  __shared__ double s_tot[kIirThreads / 32][D];
  __shared__ double s_carry[D];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t sig = blockIdx.x;
  const double* __restrict__ xs = x + sig * stride;
  double* ys = y + sig * stride;
  for (int e = tid; e < D * D * 32; e += kIirThreads) s_lane[e / 32][e % 32] = TT.lane[e % 32][(e / 32) / D * kMaxJoint + (e / 32) % D];
  if (tid < D) s_carry[tid] = zi ? zi[sig * Form::state_stride(zs) + tid] : 0.0;
  const Form form(P, TT);

  // tile `base` -> buffer: 2048 chunks of two samples, chunk c of the tile at row c / 8, column 2 (c % 8)
  auto load_tile = [&](double* buf, int64_t base) {
    const int cnt = (int)min((int64_t)kIirTile, n - base);
#pragma unroll
    for (int j = 0; j < kIirT / 2; ++j) {
      const int c = j * kIirThreads + tid;
      double* dst = buf + (c >> 3) * kJointPitch + 2 * (c & 7);
      if (kAligned) {
        const int left = cnt - 2 * c;  // samples of this chunk that exist: the rest is zero-filled
        cp_async16_zfill(dst, left > 0 ? xs + base + 2 * c : xs + base, left >= 2 ? 16 : (left == 1 ? 8 : 0));
      } else {
        dst[0] = 2 * c < cnt ? xs[base + 2 * c] : 0.0;
        dst[1] = 2 * c + 1 < cnt ? xs[base + 2 * c + 1] : 0.0;
      }
    }
  };
  if (n > 0) load_tile(s_buf0, 0);
  if (kAligned) cp_async_commit();
  __syncthreads();

  int it = 0;
  for (int64_t base = 0; base < n; base += kIirTile, ++it) {
    const int cnt = (int)min((int64_t)kIirTile, n - base);
    double* buf = (it & 1) ? s_buf1 : s_buf0;
    if (base + kIirTile < n) load_tile((it & 1) ? s_buf0 : s_buf1, base + kIirTile);
    if (kAligned) {
      cp_async_commit();
      cp_async_wait<1>();  // everything but the tile just requested has landed
    }
    __syncthreads();
    double v[kIirT];
    {
      const double2* row = reinterpret_cast<const double2*>(buf + tid * kJointPitch);
#pragma unroll
      for (int k = 0; k < kIirT / 2; ++k) {
        const double2 d = row[k];
        v[2 * k] = d.x;
        v[2 * k + 1] = d.y;
      }
    }
    const int valid = max(0, min(kIirT, cnt - tid * kIirT));  // my valid samples
    form.enter(v, valid);

    double carry[D];
#pragma unroll
    for (int i = 0; i < D; ++i) carry[i] = s_carry[i];
    // ---- pass a: end state of my chunk from the zero state (thread 0: from the tile's carry-in), state-space form
    double f[D];
#pragma unroll
    for (int i = 0; i < D; ++i) f[i] = tid == 0 ? carry[i] : 0.0;
#pragma unroll
    for (int k = 0; k < kIirT; ++k) form.state_step(v[k], f);
    // ---- scan over the threads: inclusive warp scan with constant matrices per level
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      double p[D], r[D];
#pragma unroll
      for (int i = 0; i < D; ++i) p[i] = __shfl_up_sync(0xffffffffu, f[i], 1 << d);
      if (lane >= (1 << d)) {
        double m[D * D];
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
          for (int j = 0; j < D; ++j) m[i * D + j] = TT.lvl[d][i * kMaxJoint + j];
        matvec_d<D>(m, p, r);
#pragma unroll
        for (int i = 0; i < D; ++i) f[i] += r[i];
      }
    }
    if (lane == 31) {
#pragma unroll
      for (int i = 0; i < D; ++i) s_tot[warp][i] = f[i];
    }
    double e[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      e[i] = __shfl_up_sync(0xffffffffu, f[i], 1);
      if (lane == 0) e[i] = 0.0;
    }
    __syncthreads();
    // carry entering my warp: C_w = Q C_{w-1} + tot_{w-1}, Q = (M^16)^32
    if (warp > 0) {
      double w[D], r[D], mq[D * D];
#pragma unroll
      for (int i = 0; i < D; ++i) w[i] = 0.0;
#pragma unroll
      for (int i = 0; i < D; ++i)
#pragma unroll
        for (int j = 0; j < D; ++j) mq[i * D + j] = TT.warp[i * kMaxJoint + j];
      for (int k = 0; k < warp; ++k) {
        matvec_d<D>(mq, w, r);
#pragma unroll
        for (int i = 0; i < D; ++i) w[i] = r[i] + s_tot[k][i];
      }
      double ml[D * D];
#pragma unroll
      for (int i = 0; i < D * D; ++i) ml[i] = s_lane[i][lane];
      matvec_d<D>(ml, w, r);
#pragma unroll
      for (int i = 0; i < D; ++i) e[i] += r[i];
    }
    if (tid == 0) {
#pragma unroll
      for (int i = 0; i < D; ++i) e[i] = carry[i];
    }
    // ---- pass c: the faithful recurrence from the carried-in state
    double z[D];
#pragma unroll
    for (int i = 0; i < D; ++i) z[i] = e[i];
    const bool tail_here = valid < kIirT && tid * kIirT + valid == cnt;  // the signal ends inside my chunk
    double fin[D];
#pragma unroll
    for (int i = 0; i < D; ++i) fin[i] = 0.0;
    form.filter(v, z, tail_here, valid, fin);
    form.leave(v);
    // my row back into the buffer (nobody else reads it before the barrier), then coalesced 16-byte stores
    {
      double2* row = reinterpret_cast<double2*>(buf + tid * kJointPitch);
#pragma unroll
      for (int k = 0; k < kIirT / 2; ++k) row[k] = make_double2(v[2 * k], v[2 * k + 1]);
    }
    __syncthreads();  // rows complete; all reads of s_carry / s_tot are done
    if (tail_here) {
#pragma unroll
      for (int i = 0; i < D; ++i) s_carry[i] = fin[i];
    }
    if (cnt == kIirTile && tid == kIirThreads - 1) {
#pragma unroll
      for (int i = 0; i < D; ++i) s_carry[i] = z[i];
    }
#pragma unroll
    for (int j = 0; j < kIirT / 2; ++j) {
      const int c = j * kIirThreads + tid;
      const double2 d = *reinterpret_cast<const double2*>(buf + (c >> 3) * kJointPitch + 2 * (c & 7));
      if (kAligned && 2 * c + 1 < cnt) {
        *reinterpret_cast<double2*>(ys + base + 2 * c) = d;
      } else {
        if (2 * c < cnt) ys[base + 2 * c] = d.x;
        if (2 * c + 1 < cnt) ys[base + 2 * c + 1] = d.y;
      }
    }
    __syncthreads();  // the buffer may be refilled (tile t + 2) and s_carry read (tile t + 1)
  }
  if (kAligned) cp_async_wait<0>();
  if (zf && tid < D) zf[sig * Form::state_stride(zs) + tid] = s_carry[tid];
}

// D x D matrices in long double (the scan's one-step matrix and its powers)
struct MD {
  long double m[kMaxJoint][kMaxJoint];
};
static MD md_mul(const MD& x, const MD& y, int D) {
  MD r{};
  for (int i = 0; i < D; ++i)
    for (int j = 0; j < D; ++j) {
      long double acc = 0;
      for (int k = 0; k < D; ++k) acc += x.m[i][k] * y.m[k][j];
      r.m[i][j] = acc;
    }
  return r;
}
static MD md_identity(int D) {
  MD r{};
  for (int i = 0; i < D; ++i) r.m[i][i] = 1;
  return r;
}
static void md_put(double* dst, const MD& a) {
  for (int i = 0; i < kMaxJoint; ++i)
    for (int j = 0; j < kMaxJoint; ++j) dst[i * kMaxJoint + j] = (double)a.m[i][j];
}
// (M^16)^l per lane, (M^16)^(2^d) per scan level, (M^16)^32 per warp
static void power_tables(const MD& M, int D, IirJointTables* tab) {
  MD MT = md_identity(D);
  for (int i = 0; i < kIirT; ++i) MT = md_mul(MT, M, D);
  MD pw = md_identity(D);
  for (int l = 0; l < 32; ++l) {
    md_put(tab->lane[l], pw);
    pw = md_mul(pw, MT, D);
  }
  md_put(tab->warp, pw);
  MD sq = MT;
  for (int d = 0; d < 5; ++d) {
    md_put(tab->lvl[d], sq);
    sq = md_mul(sq, sq, D);
  }
}
// homogeneous one-step matrix of the cascade: section k's input is y_{k-1} = z0_{k-1} + b0_{k-1} x_{k-1}
static void joint_tables(const IirParams& P, IirJointTables* tab) {
  const int S = P.n_sections, D = 2 * S;
  MD M{};
  for (int k = 0; k < S; ++k) {
    const long double a1 = P.sec[k].a1, a2 = P.sec[k].a2, b0 = P.sec[k].b0, b1 = P.sec[k].b1, b2 = P.sec[k].b2;
    const long double c1 = b1 - a1 * b0, c2 = b2 - a2 * b0;
    tab->c[2 * k] = (double)c1;
    tab->c[2 * k + 1] = (double)c2;
    M.m[2 * k][2 * k] = -a1;
    M.m[2 * k][2 * k + 1] = 1;
    M.m[2 * k + 1][2 * k] = -a2;
    // the input of section k as a linear function of the earlier sections' states (x = 0): u_k = z0_{k-1} + b0_{k-1} u_{k-1}
    long double gain = 1;
    for (int j = k - 1; j >= 0; --j) {
      M.m[2 * k][2 * j] += c1 * gain;
      M.m[2 * k + 1][2 * j] += c2 * gain;
      gain *= P.sec[j].b0;
    }
  }
  power_tables(M, D, tab);
}
// one-step matrix of lfilter's DF2T state (order Mo): z_i' = -a_{i+1} z_0 + z_{i+1}
static void lfilter_tables(const LfilterParams& P, IirJointTables* tab) {
  const int Mo = P.order;
  MD M{};
  for (int i = 0; i < Mo; ++i) {
    tab->c[i] = (double)((long double)P.b[i + 1] - (long double)P.a[i + 1] * (long double)P.b[0]);
    M.m[i][0] = -(long double)P.a[i + 1];
    if (i + 1 < Mo) M.m[i][i + 1] = 1;
  }
  power_tables(M, Mo, tab);
}

// The scan kernel of Form<k> (k = sections or order, 1..Form::kMax) over n_sig signals, with 16-byte accesses when
// every row of x and y starts on a 16-byte boundary.
template <template <int> class Form, int K = 1>
static cudaError_t launch_scan(int k, const typename Form<K>::Params& P, const IirJointTables& T, const double* x,
                               double* y, int64_t n_sig, int64_t n, int64_t stride, const double* zi, double* zf,
                               int zs, cudaStream_t st) {
  if constexpr (K < Form<K>::kMax) {
    if (k > K) return launch_scan<Form, K + 1>(k, P, T, x, y, n_sig, n, stride, zi, zf, zs, st);
  }
  const bool aligned = ((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0) && (stride % 2 == 0 || n_sig == 1);
  const auto kern = aligned ? iir_scan_kernel<Form<K>, true> : iir_scan_kernel<Form<K>, false>;
  const int smem = 2 * kJointTileBytes;
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)n_sig, kIirThreads, smem, st>>>(P, T, x, y, n, stride, zi, zf, zs);
  return cudaGetLastError();
}

// Host -> device copy of a small table (the initial states) that does NOT stall the stream: cudaMemcpyAsync from
// PAGEABLE memory synchronises the stream before it stages the data, which serialises the host with every filter call
// (predistort in scan mode: 0.32 ms of kernel became 0.59 ms per call).  The bytes go through a small ring of pinned
// buffers per host thread instead; a slot is reused only after the copy that read it has completed (one event each).
static cudaError_t upload_small(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  constexpr int kSlots = 4;
  constexpr size_t kSlotBytes = 64 << 10;
  struct Ring {
    unsigned char* host[kSlots] = {};
    cudaEvent_t done[kSlots] = {};
    int next = 0;
  };
  static thread_local Ring rings[64];  // per host thread AND device: an event belongs to the device it was created on
  if (bytes == 0) return cudaSuccess;
  int dev = -1;
  if (bytes > kSlotBytes || cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
  Ring& ring = rings[dev];
  const int i = ring.next;
  cudaError_t e = cudaSuccess;
  if (!ring.host[i]) {
    e = cudaHostAlloc((void**)&ring.host[i], kSlotBytes, cudaHostAllocPortable);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ring.done[i], cudaEventDisableTiming);
    if (e != cudaSuccess) {
      cudaGetLastError();
      ring.host[i] = nullptr;
      return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
    }
  } else {
    e = cudaEventSynchronize(ring.done[i]);
    if (e != cudaSuccess) return e;
  }
  memcpy(ring.host[i], src, bytes);
  e = cudaMemcpyAsync(dst, ring.host[i], bytes, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaEventRecord(ring.done[i], st);
  ring.next = (i + 1) % kSlots;
  return e;
}

// One filter call's states on the device: `words` doubles of HOST zi / zf (either may be NULL) in stream-ordered
// scratch, zi uploaded, then run(d_zi, d_zf) filters; zf is copied back and the stream synchronised before the call
// returns, because the caller reads zf then.  An empty signal (n = 0) passes the state through: zf = zi, or zeros
// without zi.
template <class Run>
static int with_states(const double* zi, double* zf, size_t words, int64_t n, cudaStream_t st, Run run) {
  const size_t bytes = sizeof(double) * words;
  double *d_zi = nullptr, *d_zf = nullptr;
  cudaError_t e = cudaSuccess;
  if (zi && words) {
    e = cudaMallocAsync(&d_zi, bytes, st);
    if (e == cudaSuccess) e = upload_small(d_zi, zi, bytes, st);
  }
  if (e == cudaSuccess && zf && words) e = cudaMallocAsync(&d_zf, bytes, st);
  if (e == cudaSuccess && n > 0) {
    e = run(d_zi, d_zf);
  } else if (e == cudaSuccess && d_zf) {
    e = d_zi ? cudaMemcpyAsync(d_zf, d_zi, bytes, cudaMemcpyDeviceToDevice, st) : cudaMemsetAsync(d_zf, 0, bytes, st);
  }
  if (e == cudaSuccess && d_zf) {
    e = cudaMemcpyAsync(zf, d_zf, bytes, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  if (d_zi) cudaFreeAsync(d_zi, st);
  if (d_zf) cudaFreeAsync(d_zf, st);
  return e == cudaSuccess ? WFM_OK : WFM_ECUDA;
}

}  // namespace wfm

extern "C" int wfm_sosfilt(const double* sos, int32_t n_sections, double initial, const double* x, double* y,
                           int64_t n_sig, int64_t n, int64_t stride, const double* zi, double* zf, int32_t mode,
                           void* stream) {
  using namespace wfm;
  if (!sos || n_sections < 1 || n_sections > kMaxSections || n_sig < 0 || n < 0 || (n_sig > 1 && stride < n))
    return WFM_EINVAL;
  if (mode != WFM_IIR_EXACT && mode != WFM_IIR_SCAN) return WFM_EINVAL;
  if (n_sig == 0) return WFM_OK;
  if ((!x || !y) && n > 0) return WFM_EINVAL;  // (an empty signal has no buffer to point at)
  cudaStream_t st = (cudaStream_t)stream;
  IirParams P{};
  P.n_sections = n_sections;
  P.initial = initial;
  for (int k = 0; k < n_sections; ++k) {
    const double* c = sos + 6 * k;
    const double a0 = c[3];
    // scipy normalises by a0 when it is not 1
    P.sec[k] = {c[0] / a0, c[1] / a0, c[2] / a0, c[4] / a0, c[5] / a0};
  }
  return with_states(zi, zf, 2 * (size_t)n_sections * (size_t)n_sig, n, st, [&](const double* d_zi, double* d_zf) {
    if (mode == WFM_IIR_EXACT) {
      const unsigned blocks = (unsigned)((n_sig + kExactWarps - 1) / kExactWarps);
      sosfilt_exact_kernel<<<blocks, 32 * kExactWarps, 0, st>>>(P, x, y, n_sig, n, stride, d_zi, d_zf);
      return cudaGetLastError();
    }
    // the scan takes the sections two by two: a cascade of S sections is ceil(S / 2) launches, each a read and a write
    // of the signal; `initial` is subtracted by the first launch and added back by the last one only
    cudaError_t e = cudaSuccess;
    for (int k0 = 0; k0 < n_sections && e == cudaSuccess; k0 += 2) {
      IirParams Pk{};
      Pk.n_sections = std::min(2, n_sections - k0);
      Pk.initial = P.initial;
      Pk.shift_in = k0 == 0;
      Pk.shift_out = k0 + 2 >= n_sections;
      for (int k = 0; k < Pk.n_sections; ++k) Pk.sec[k] = P.sec[k0 + k];
      static thread_local IirJointTables jt;
      joint_tables(Pk, &jt);
      e = launch_scan<BiquadForm>(Pk.n_sections, Pk, jt, k0 == 0 ? x : y, y, n_sig, n, stride,
                                  d_zi ? d_zi + 2 * k0 : nullptr, d_zf ? d_zf + 2 * k0 : nullptr, 2 * n_sections, st);
    }
    return e;
  });
}

extern "C" int wfm_lfilter(const double* b, int32_t nb, const double* a, int32_t na, const double* x, double* y,
                           int64_t n_sig, int64_t n, int64_t stride, const double* zi, double* zf, void* stream) {
  return wfm_lfilter_mode(b, nb, a, na, x, y, n_sig, n, stride, zi, zf, WFM_IIR_EXACT, stream);
}

extern "C" int wfm_lfilter_mode(const double* b, int32_t nb, const double* a, int32_t na, const double* x, double* y,
                                int64_t n_sig, int64_t n, int64_t stride, const double* zi, double* zf, int32_t mode,
                                void* stream) {
  using namespace wfm;
  if (mode != WFM_IIR_EXACT && mode != WFM_IIR_SCAN) return WFM_EINVAL;
  if (!b || !a || nb < 1 || na < 1 || a[0] == 0.0 || n_sig < 0 || n < 0 || (n_sig > 1 && stride < n)) return WFM_EINVAL;
  const int M = std::max(nb, na) - 1;
  if (M > kMaxOrder) return WFM_EUNSUPPORTED;
  if (n_sig == 0) return WFM_OK;
  if ((!x || !y) && n > 0) return WFM_EINVAL;  // (an empty signal has no buffer to point at)
  cudaStream_t st = (cudaStream_t)stream;
  LfilterParams P{};
  P.order = M;
  for (int k = 0; k <= M; ++k) {  // scipy normalises both polynomials by a[0]
    P.b[k] = k < nb ? b[k] / a[0] : 0.0;
    P.a[k] = k < na ? a[k] / a[0] : 0.0;
  }
  return with_states(zi, zf, (size_t)M * (size_t)n_sig, n, st, [&](const double* d_zi, double* d_zf) {
    if (mode == WFM_IIR_SCAN && M >= 1 && M <= kMaxJoint) {
      static thread_local IirJointTables jt;
      lfilter_tables(P, &jt);
      return launch_scan<DirectForm>(M, P, jt, x, y, n_sig, n, stride, d_zi, d_zf, M, st);
    }
    // (orders above 4 and order 0: the sequential kernel, whatever the mode)
    lfilter_exact_kernel<<<(unsigned)((n_sig + kExactWarps - 1) / kExactWarps), 32 * kExactWarps, 0, st>>>(
        P, x, y, n_sig, n, stride, d_zi, d_zf);
    return cudaGetLastError();
  });
}
