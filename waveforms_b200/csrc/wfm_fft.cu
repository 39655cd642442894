// wfm_fft.cu — K3: hand-written shared-memory Stockham FFT (fp64 complex) and the
// frequency-domain filter built on it.  No cuFFT.
//
// Replaces np.fft.fft / np.fft.ifft in
// /root/reference/waveforms/distortion.py:208-221 (reflection,
// correct_reflection: y = ifft(fft(x) * H).real on the np.fft.fftfreq grid) and
// scipy.signal.fftconvolve in distortion.py:329-333 (predistort with a kernel),
// for ARBITRARY n (config 4: n = 400 000 = 2^7 * 5^5).
//
// Building block: `smem_fft` — C interleaved length-L transforms resident in
// shared memory, mixed-radix Stockham autosort (radices 7,5,3,10,8,4,2), ping-pong
// between two buffers.  Twiddles: ONE look-up per butterfly, W^k from a compact
// per-stage table (host, long double), the powers W^(k r) formed in registers — the
// row pass saturates the shared-memory pipe, not the FP64 pipe.  `smem_fft_ct` is the
// same transform with the whole plan as template arguments (625 = 5^4 x 4 columns,
// 640 = 10 x 8 x 8 x 2 rows / 4 columns: the tile shapes of cfg4).
//
//   n <= kMaxPoints, 7-smooth     one CTA per signal:
//                                 load real -> FFT_n -> xH -> IFFT_n -> store real
//   n = N1*N2 (both <= kMaxPoints, 7-smooth)   four-step, three kernels:
//        A  column FFTs of length N1 (tiles of C columns), twiddle W_n^(n2 k1),
//           real in -> complex scratch  [k1][n2]
//        B  row FFT_N2 -> x H[k1 + N1 k2] -> row IFFT_N2, in place in scratch
//           (fft_rows_tma_kernel: rows and response rows land by cp.async.bulk,
//           leave by bulk stores).  The spectrum is never brought to natural order:
//           H is permuted once instead, which saves two transposes.
//        C  conj twiddle, column IFFT_N1, scale 1/n, real part -> output
//   otherwise (a prime factor > 7)   Bluestein: chirp-z through 7-smooth
//        transforms of length M >= 2n-1 (generic c2c path).
//
// Two real signals ride one complex transform (the response is made Hermitian), so
// the HBM traffic of the fused path is 8+8 (A), 8+8 (B), 8+8 (C) = 48 B per real
// sample (SURVEY 8d counts 16 B for an ideal single pass).
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <complex>
#include <cstdint>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>
#include "wfm_internal.h"

namespace wfm {

// ---- tile geometry: fixed, every alternative below was measured on cfg4 and rejected (DESIGN §K3) --------------------
// Radices: the largest power-of-two butterfly is 8 (4 / 8 / 16: 6.11 / 5.90 / 6.30 ms); the one composite butterfly
// is 10 = 2 x 5 (25 = 5 x 5 in the column passes: 2.19-2.20 against 2.19 ms).  The shared-memory buffers are unpadded
// (a 16-byte pad per 32 / 16 elements: 2.24 / 2.26 against 2.20 ms: the reads pay what the writes gain), and the
// transform direction is a run-time argument of the stages (compile-time: 2.21 against 2.19 ms).
constexpr int kFftThreads = 512;  // one-level kernels: one CTA per transform
// the row pass has the radix-10 stage and reads contiguous rows, so its tile can be small: 2 rows per CTA, 160 threads
// (the 160 radix-8 / 128 radix-10 butterflies of a 640-point x 2 tile), three CTAs per SM at up to 136 registers.  More,
// smaller CTAs overlap the load / butterfly / store phases that block barriers serialise inside one CTA.  Measured on
// cfg4 (fft_filter, ms): 4 rows x 320 threads x 2 CTAs 2.19 (512 / 448 / 384 threads: 2.27 / 2.21 / 2.20);
// 2 rows x 160 x 3 CTAs 2.08; x 4 CTAs 2.13; x 2 CTAs 2.24; 2 rows x 128 x 3: 2.16; x 192 x 3: 2.12; 1 row x 96 x 6: 2.19
constexpr int kFftRowsThreads = 160;
constexpr int kFftRowsMinBlocks = 3;
constexpr int kFftRowsLogC = 1;
// column pass: 4 interleaved columns per CTA and two CTAs per SM (32 warps) measured 14 % faster than 8 columns and one
// CTA (cfg4, n = 625 x 640)
constexpr int kFftColsThreads = 512;
constexpr int kFftColsMinBlocks = 2;
constexpr int kFftColsLogC = 2;
constexpr int kMaxPoints = 6144;  // complex points per shared-memory buffer (2 buffers = 192 KB)
constexpr int kMaxStages = 20;
constexpr int kSmemBudget = 227 * 1024 - 1024;
constexpr int kPlanSlackBytes = 1024;  // behind the buffers and the twiddle table: per-column inter-pass twiddles of a tile

struct FftPlan {
  int L;
  int n_stage;
  int radix[kMaxStages];
  uint32_t inv_ns[kMaxStages];  // ceil(2^32 / Ns) of every stage: j / Ns = umulhi(j, inv) for j < 2^16
  int twc_len;         // entries of twc: sum of the stage strides Ns
  const double2* twc;  // compact per-stage twiddle table (global memory): for stage s (stride Ns = product of the earlier
                       // radices) the Ns values exp(-2 pi i k / (Ns R_s)), k < Ns, back to back; long double on the host
  int tw_in_smem;     // the kernels stage the table in shared memory behind the two buffers (an area of L entries)
};

__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
  return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ double2 cscale(double2 a, double s) { return make_double2(a.x * s, a.y * s); }
// multiply by sgn*i  (sgn = +1: i*a; sgn = -1: -i*a)
__device__ __forceinline__ double2 cmul_i(double2 a, double sgn) { return make_double2(-sgn * a.y, sgn * a.x); }

template <int R>
__device__ __forceinline__ void dft_small(double2 (&v)[R], double sgn);  // sgn = -1 forward, +1 inverse

template <>
__device__ __forceinline__ void dft_small<2>(double2 (&v)[2], double) {
  double2 a = v[0], b = v[1];
  v[0] = cadd(a, b);
  v[1] = csub(a, b);
}
template <>
__device__ __forceinline__ void dft_small<3>(double2 (&v)[3], double sgn) {
  const double h = 0.86602540378443864676;  // sqrt(3)/2
  double2 s = cadd(v[1], v[2]), d = csub(v[1], v[2]);
  double2 m = make_double2(v[0].x - 0.5 * s.x, v[0].y - 0.5 * s.y);
  double2 r = cmul_i(cscale(d, h), sgn);
  v[0] = cadd(v[0], s);
  v[1] = cadd(m, r);
  v[2] = csub(m, r);
}
template <>
__device__ __forceinline__ void dft_small<4>(double2 (&v)[4], double sgn) {
  double2 t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
  double2 t2 = cadd(v[1], v[3]), t3 = cmul_i(csub(v[1], v[3]), sgn);
  v[0] = cadd(t0, t2);
  v[1] = cadd(t1, t3);
  v[2] = csub(t0, t2);
  v[3] = csub(t1, t3);
}
template <>
__device__ __forceinline__ void dft_small<5>(double2 (&v)[5], double sgn) {
  const double c1 = 0.30901699437494742410, c2 = -0.80901699437494742410;
  const double s1 = 0.95105651629515357212, s2 = 0.58778525229247312917;
  double2 a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
  double2 b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
  double2 t1 = make_double2(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
  double2 t2 = make_double2(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
  double2 u1 = cmul_i(make_double2(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y), sgn);
  double2 u2 = cmul_i(make_double2(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y), sgn);
  v[0] = cadd(v[0], cadd(a1, a2));
  v[1] = cadd(t1, u1);
  v[4] = csub(t1, u1);
  v[2] = cadd(t2, u2);
  v[3] = csub(t2, u2);
}
template <>
__device__ __forceinline__ void dft_small<7>(double2 (&v)[7], double sgn) {
  const double c[7] = {1.0, 0.62348980185873353053, -0.22252093395631440429, -0.90096886790241912624,
                       -0.90096886790241912624, -0.22252093395631440429, 0.62348980185873353053};
  const double s[7] = {0.0, 0.78183148246802980871, 0.97492791218182360702, 0.43388373911755812048,
                       -0.43388373911755812048, -0.97492791218182360702, -0.78183148246802980871};
  double2 o[7];
#pragma unroll
  for (int p = 0; p < 7; ++p) {
    double2 acc = v[0];
#pragma unroll
    for (int q = 1; q < 7; ++q) {
      const int m = (p * q) % 7;
      acc = cadd(acc, cmul(v[q], make_double2(c[m], sgn * s[m])));
    }
    o[p] = acc;
  }
#pragma unroll
  for (int p = 0; p < 7; ++p) v[p] = o[p];
}

// R = R1*R2 point DFT in registers (Cooley-Tukey inside the thread): input index n = n1 + R1*n2,
// output index k = R2*k1 + k2; cs/sn hold cos / sin of 2 pi m / R.  Fully unrolled: every index is a
// compile-time constant, so v stays in registers.
template <int R1, int R2>
__device__ __forceinline__ void dft_composite(double2 (&v)[R1 * R2], double sgn, const double* cs, const double* sn) {
  constexpr int R = R1 * R2;
  double2 y[R];
#pragma unroll
  for (int n1 = 0; n1 < R1; ++n1) {
    double2 t[R2];
#pragma unroll
    for (int n2 = 0; n2 < R2; ++n2) t[n2] = v[n1 + R1 * n2];
    dft_small<R2>(t, sgn);
#pragma unroll
    for (int k2 = 0; k2 < R2; ++k2) {
      const int m = (n1 * k2) % R;
      y[n1 * R2 + k2] = m == 0 ? t[k2] : cmul(t[k2], make_double2(cs[m], sgn * sn[m]));
    }
  }
#pragma unroll
  for (int k2 = 0; k2 < R2; ++k2) {
    double2 t[R1];
#pragma unroll
    for (int n1 = 0; n1 < R1; ++n1) t[n1] = y[n1 * R2 + k2];
    dft_small<R1>(t, sgn);
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) v[R2 * k1 + k2] = t[k1];
  }
}
template <>
__device__ __forceinline__ void dft_small<8>(double2 (&v)[8], double sgn) {
  constexpr double cs[8] = {1.0, 0.7071067811865476, 6.123233995736766e-17, -0.7071067811865475, -1.0, -0.7071067811865477, -1.8369701987210297e-16, 0.7071067811865474};
  constexpr double sn[8] = {0.0, 0.7071067811865475, 1.0, 0.7071067811865476, 1.2246467991473532e-16, -0.7071067811865475, -1.0, -0.7071067811865477};
  dft_composite<2, 4>(v, sgn, cs, sn);
}
template <>
__device__ __forceinline__ void dft_small<10>(double2 (&v)[10], double sgn) {
  constexpr double cs[10] = {1.0, 0.8090169943749475, 0.30901699437494745, -0.30901699437494734, -0.8090169943749473, -1.0, -0.8090169943749476, -0.30901699437494756, 0.30901699437494723, 0.8090169943749473};
  constexpr double sn[10] = {0.0, 0.5877852522924731, 0.9510565162951535, 0.9510565162951536, 0.5877852522924732, 1.2246467991473532e-16, -0.587785252292473, -0.9510565162951535, -0.9510565162951536, -0.5877852522924734};
  dft_composite<2, 5>(v, sgn, cs, sn);
}

// ---- Stockham stages ------------------------------------------------------------------
// C = 2^logc interleaved transforms live in shared memory, point p of transform c at
// [p*C + c].  A stage reads its R inputs through `in(p, c, e)` and hands its R outputs to
// `out(p, c, e, v)`, e = (p << logc) + c the element's index in a shared-memory buffer: the
// middle stages use the shared-memory accessors below, the FIRST stage of a transform reads
// global memory directly and the LAST one writes global memory (or multiplies by the response
// on the way to shared memory), so loading, filtering and storing cost no passes of their own
// over shared memory — the shared-memory data pipe is what bounds these kernels (ncu: 75 % of
// its peak, profiles/r1o_k3_ncu_details.txt).  An accessor uses what it needs of (p, c, e).
// accessors that have no inter-pass twiddle carry this no-op (a member, so they stay aggregates)
#define WFM_NO_RUN_TWIDDLE \
  template <int R>         \
  __device__ __forceinline__ void twiddle_run(double2 (&)[R], int, int, int) const {}
struct SmemIn {
  WFM_NO_RUN_TWIDDLE
  const double2* a;
  __device__ __forceinline__ double2 operator()(int, int, int e) const { return a[e]; }
};
struct SmemOut {
  WFM_NO_RUN_TWIDDLE
  double2* b;
  __device__ __forceinline__ void operator()(int, int, int e, double2 v) const { b[e] = v; }
};

// twiddles W^(k r), r = 1..R-1, of one butterfly: ONE look-up, W^k from the stage's slice of the compact table
// (FftPlan.twc: consecutive k at consecutive addresses — in a full W_L^p table a stage's twiddles sit L / (Ns R) * 16
// bytes apart, a multiple of the bank period for the early stages of even lengths: up to 16-way conflicts), the powers by
// products of depth <= log2 R (a few roundings more; the FP64 pipe idles in these kernels, the shared-memory pipe does not)
template <int R>
__device__ __forceinline__ void load_twiddles(double2 (&w)[R], const double2* __restrict__ tw_k, double sgn) {
  w[1] = *tw_k;
  w[1].y *= -sgn;  // table holds exp(-i..): forward (sgn=-1) keeps it, inverse conjugates
#pragma unroll
  for (int r = 2; r < R; ++r) w[r] = (r & 1) ? cmul(w[r - 1], w[1]) : cmul(w[r / 2], w[r / 2]);
}

template <int R, class In, class Out>
__device__ __forceinline__ void stockham_stage(In in, Out out, int L, int logc, int Ns, uint32_t inv_ns, int toff,
                                               const double2* __restrict__ tw, double sgn) {
  const int nb = L / R;        // butterflies per transform; toff: where the stage's Ns twiddles start in the compact table
  const int cmask = (1 << logc) - 1;
  const int total = nb << logc;
  for (int jj = threadIdx.x; jj < total; jj += blockDim.x) {
    const int c = jj & cmask, j = jj >> logc;
    const int q = Ns == 1 ? j : (int)__umulhi((uint32_t)j, inv_ns);  // j / Ns
    const int k = j - q * Ns;
    double2 v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = in(j + r * nb, c, ((j + r * nb) << logc) + c);
    in.template twiddle_run<R>(v, j, nb, c);  // inter-pass twiddles of the run j, j+nb, ... (column passes)
    if (k > 0) {
      double2 w[R];
      load_twiddles<R>(w, tw + toff + k, sgn);
#pragma unroll
      for (int r = 1; r < R; ++r) v[r] = cmul(v[r], w[r]);
    }
    dft_small<R>(v, sgn);
    const int j0 = q * Ns * R + k;
    out.template twiddle_run<R>(v, j0, Ns, c);
#pragma unroll
    for (int r = 0; r < R; ++r) out(j0 + r * Ns, c, ((j0 + r * Ns) << logc) + c, v[r]);
  }
}

template <class In, class Out>
__device__ __forceinline__ void stage_any(int R, In in, Out out, int L, int logc, int Ns, uint32_t inv, int toff,
                                          const double2* __restrict__ tw, double sgn) {
  switch (R) {
    case 2: stockham_stage<2>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    case 3: stockham_stage<3>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    case 4: stockham_stage<4>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    case 5: stockham_stage<5>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    case 8: stockham_stage<8>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    case 10: stockham_stage<10>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
    default: stockham_stage<7>(in, out, L, logc, Ns, inv, toff, tw, sgn); break;
  }
}

// One length-P.L transform of C = 2^logc interleaved signals.  Stage 0 reads through `in`
// and writes buf0; stage s >= 1 reads buf[(s-1)&1] and writes buf[s&1]; the last stage
// writes through `out` instead.  `in` may read buf1 (never buf0).  Ends with a block
// barrier, so what `out` wrote to shared memory is visible.  All threads must call it.
template <class In, class Out>
__device__ __forceinline__ void smem_fft(const FftPlan& P, int logc, double sgn, const double2* __restrict__ tw, In in,
                                         Out out, double2* buf0, double2* buf1) {
  const int S = P.n_stage;
  if (S == 0) {  // L == 1: the transform is the identity
    for (int c = threadIdx.x; c < (1 << logc); c += blockDim.x) out(0, c, c, in(0, c, c));
    __syncthreads();
    return;
  }
  if (S == 1) {
    stage_any(P.radix[0], in, out, P.L, logc, 1, P.inv_ns[0], 0, tw, sgn);
    __syncthreads();
    return;
  }
  stage_any(P.radix[0], in, SmemOut{buf0}, P.L, logc, 1, P.inv_ns[0], 0, tw, sgn);
  __syncthreads();
  int Ns = P.radix[0], toff = 1;
  double2 *src = buf0, *dst = buf1;
  for (int s = 1; s < S - 1; ++s) {
    stage_any(P.radix[s], SmemIn{src}, SmemOut{dst}, P.L, logc, Ns, P.inv_ns[s], toff, tw, sgn);
    __syncthreads();
    double2* t = src; src = dst; dst = t;
    toff += Ns;
    Ns *= P.radix[s];
  }
  stage_any(P.radix[S - 1], SmemIn{src}, out, P.L, logc, Ns, P.inv_ns[S - 1], toff, tw, sgn);
  __syncthreads();
}
// the buffer the last stage of smem_fft(.., buf0, buf1) may write through `out` (the one it
// does not read)
__device__ __forceinline__ double2* last_stage_target(const FftPlan& P, double2* buf0, double2* buf1) {
  return ((P.n_stage - 1) & 1) ? buf1 : buf0;
}

// the plan's twiddle table: staged behind the two ping-pong buffers when it fits
__device__ __forceinline__ const double2* stage_twiddles(const FftPlan& P, double2* smem_after_buffers) {
  if (!P.tw_in_smem) return P.twc;
  for (int p = threadIdx.x; p < P.twc_len; p += blockDim.x) smem_after_buffers[p] = P.twc[p];
  return smem_after_buffers;  // visible after the caller's next __syncthreads()
}

// Inter-pass twiddles W_n^m = exp(-2 pi i m / n), 0 <= m < n, from two small host tables
// (long double): m = 1024 h + l, W^m = hi[h] * lo[l].  One complex multiply instead of a
// sincospi per element; the 1024 + n/1024 entries stay in L1.
struct BigTwiddle {
  const double2* hi;  // W_n^(1024 h)
  const double2* lo;  // W_n^l, l < 1024
};
__device__ __forceinline__ double2 big_twiddle(const BigTwiddle& T, int64_t m, double sgn) {
  double2 w = cmul(__ldg(T.hi + (m >> 10)), __ldg(T.lo + (m & 1023)));
  w.y *= -sgn;  // tables hold exp(-i ..): forward (sgn = -1) keeps it, inverse conjugates
  return w;
}

extern __shared__ __align__(16) unsigned char fft_smem_raw[];

// ---- one-level fused filter: n <= kMaxPoints -------------------------------------
// One CTA per PAIR of real signals: z = x_a + i x_b goes through one complex transform.  H is
// the Hermitian part of the caller's response (hermitian_part_kernel), so ifft(fft(z) H) =
// y_a + i y_b with both real.
// nv: samples the signals really hold (<= transform length): reads beyond are zeros, writes beyond are dropped — the
// zero padding of a linear convolution costs no pass over memory
struct PairIn {
  WFM_NO_RUN_TWIDDLE  // two real signals -> one complex
  const double* xa;
  const double* xb;  // nullptr: odd tail
  int nv;
  __device__ __forceinline__ double2 operator()(int p, int, int) const {
    return p < nv ? make_double2(xa[p], xb ? xb[p] : 0.0) : make_double2(0.0, 0.0);
  }
};
struct PairOut {
  WFM_NO_RUN_TWIDDLE
  double* ya;
  double* yb;
  double scale;
  int nv;
  __device__ __forceinline__ void operator()(int p, int, int, double2 v) const {
    if (p >= nv) return;
    ya[p] = v.x * scale;
    if (yb) yb[p] = v.y * scale;
  }
};
struct MulHOut {
  WFM_NO_RUN_TWIDDLE  // spectrum x response on the way to shared memory
  double2* z;
  const double2* __restrict__ H;
  __device__ __forceinline__ void operator()(int p, int, int, double2 v) const { z[p] = cmul(v, __ldg(H + p)); }
};
__global__ void __launch_bounds__(kFftThreads) fft_filter_single_kernel(FftPlan P, const double* __restrict__ x,
                                                                        double* __restrict__ y, int64_t stride,
                                                                        int64_t y_stride, int64_t n_sig,
                                                                        const double2* __restrict__ H, int nv) {
  double2* a = reinterpret_cast<double2*>(fft_smem_raw);
  double2* b = a + P.L;
  const double2* tw = stage_twiddles(P, b + P.L);
  const int64_t s0 = 2 * (int64_t)blockIdx.x;
  const bool two = s0 + 1 < n_sig;
  const double* xs = x + s0 * stride;
  double* ys = y + s0 * y_stride;
  double2* z = last_stage_target(P, a, b);
  smem_fft(P, 0, -1.0, tw, PairIn{xs, two ? xs + stride : nullptr, nv}, MulHOut{z, H}, a, b);
  smem_fft(P, 0, +1.0, tw, SmemIn{z}, PairOut{ys, two ? ys + y_stride : nullptr, 1.0 / (double)P.L, nv}, z == a ? b : a, z);
}

// ---- compile-time plans -------------------------------------------------------------------------------------------------
// The generic stages take the transform length, the interleave, the radix sequence and the strides at run time: two
// thirds of their instructions are index arithmetic (ncu: 88 M fp64 of 365 M warp instructions per column pass of cfg4).
// For the tile shapes that matter the whole plan is a template argument: element indices become immediate offsets, the
// butterfly count per thread is a constant, j / Ns is a multiply-shift by a constant.  The accessors are those of the
// generic stages.  The inverse twiddle product conjugates inside its fma arrangement, where stockham_stage conjugates W
// and calls cmul: the two round differently in the last bit, so the two stage bodies stay separate.
template <int R, int L, int LOGC, int NS, int TOFF, bool kFwd, int T, class In, class Out>
__device__ __forceinline__ void stage_ct(In in, Out out, const double2* __restrict__ tw) {
  constexpr double sgn = kFwd ? -1.0 : 1.0;
  constexpr int nb = L / R, nbC = nb << LOGC, NsC = NS << LOGC;
  constexpr int iters = (nbC + T - 1) / T;
#pragma unroll
  for (int it = 0; it < iters; ++it) {
    const int jj = (int)threadIdx.x + it * T;
    if (nbC % T != 0 && jj >= nbC) break;
    const int c = jj & ((1 << LOGC) - 1), j = jj >> LOGC;
    const int q = NS == 1 ? j : j / NS;
    const int k = j - q * NS;
    double2 v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = in(j + r * nb, c, jj + r * nbC);
    in.template twiddle_run<R>(v, j, nb, c);
    if (NS > 1 && k > 0) {
      // ONE look-up per butterfly, W^k from the stage's own compact table (consecutive k: consecutive addresses, no bank
      // conflicts — in the full table a stage's twiddles are L / (NS R) * 16 bytes apart, a multiple of the 128-byte bank
      // period for the early stages); W^(k r) by products of depth <= 3.  The shared-memory pipe, not the FP64 pipe, is
      // what these passes saturate.
      double2 w[R];
      w[1] = tw[TOFF + k];
#pragma unroll
      for (int r = 2; r < R; ++r) w[r] = (r & 1) ? cmul(w[r - 1], w[1]) : cmul(w[r / 2], w[r / 2]);
#pragma unroll
      for (int r = 1; r < R; ++r)
        v[r] = kFwd ? make_double2(fma(v[r].x, w[r].x, -v[r].y * w[r].y), fma(v[r].x, w[r].y, v[r].y * w[r].x))
                    : make_double2(fma(v[r].x, w[r].x, v[r].y * w[r].y), fma(v[r].y, w[r].x, -v[r].x * w[r].y));
    }
    dft_small<R>(v, sgn);
    const int j0 = j + q * (NS * (R - 1));
    const int e0 = jj + q * (NsC * (R - 1));
    out.template twiddle_run<R>(v, j0, NS, c);
#pragma unroll
    for (int r = 0; r < R; ++r) out(j0 + r * NS, c, e0 + r * NsC, v[r]);
  }
}
// stages 0 .. S-1 of the radix pack; stage s reads `in` (s = 0) or the buffer stage s-1 wrote, and writes `out`
// (s = S-1) or buf[s & 1]
struct CtNoHook {
  __device__ __forceinline__ void operator()() const {}
};
// `hook` runs once, after the first stage's butterflies and before its barrier: shared-memory stores placed there (tables
// whose global loads were issued before the stage) are visible to every later stage at no extra barrier
template <int L, int LOGC, bool kFwd, int T, int NS, int TOFF, class In, class Out, class Hook, int R0, int... Rest>
__device__ __forceinline__ void stages_ct_impl(int s, In in, Out out, const double2* __restrict__ tw, double2* buf0, double2* buf1,
                                               Hook hook, std::integer_sequence<int, R0, Rest...>) {
  double2* dst = (s & 1) ? buf1 : buf0;
  if constexpr (sizeof...(Rest) == 0) {
    stage_ct<R0, L, LOGC, NS, TOFF, kFwd, T>(in, out, tw);
    hook();
    __syncthreads();
  } else {
    stage_ct<R0, L, LOGC, NS, TOFF, kFwd, T>(in, SmemOut{dst}, tw);
    hook();
    __syncthreads();
    stages_ct_impl<L, LOGC, kFwd, T, NS * R0, TOFF + NS>(s + 1, SmemIn{dst}, out, tw, buf0, buf1, CtNoHook{},
                                                         std::integer_sequence<int, Rest...>{});
  }
}
// same contract as smem_fft: `in` may read buf1, the last stage writes through `out` (last_stage_target is the buffer it
// does not read).  The transform length is the product of the radices.
template <int LOGC, bool kFwd, int T, int... Rs, class In, class Out, class Hook = CtNoHook>
__device__ __forceinline__ void smem_fft_ct(std::integer_sequence<int, Rs...> radices, In in, Out out,
                                            const double2* __restrict__ tw, double2* buf0, double2* buf1, Hook hook = Hook{}) {
  stages_ct_impl<(Rs * ...), LOGC, kFwd, T, 1, 0>(0, in, out, tw, buf0, buf1, hook, radices);
}
// the compile-time plans: 625 = 5^4 (column passes of n = 400 000) and 640 = 10 x 8 x 8 (the passes of n = 409 600)
using Radices625 = std::integer_sequence<int, 5, 5, 5, 5>;
using Radices640 = std::integer_sequence<int, 10, 8, 8>;
// entries of a plan's compact twiddle table: the sum of the stage strides 1, R0, R0 R1, ...
template <int... Rs>
__host__ __device__ constexpr int ct_twiddle_count(std::integer_sequence<int, Rs...>) {
  int n = 0, ns = 1;
  ((n += ns, ns *= Rs), ...);
  return n;
}
// stride of a plan's last stage: L / last radix
template <int... Rs>
__host__ __device__ constexpr int ct_last_stride(std::integer_sequence<int, Rs...>) {
  int ns = 1, last = 1;
  ((ns *= Rs, last = Rs), ...);
  return ns / last;
}

// ---- four-step, kernel A / C: column transforms of length N1 -----------------------
// element (r, n2) of the [N1][N2] view; C = 2^logc adjacent columns per CTA.  The inter-pass
// twiddle W_n^(sgn * r * n2) (r * n2 < n: no reduction needed) is applied after the
// transform (first pass of a forward-structured transform) or before it (last pass of the
// fused filter, undoing the forward pass)
// kRealIn / kRealOut: the signal index is a PAIR of real signals packed as the real and
// imaginary part of one complex signal (the filter's response is Hermitian); pb == nullptr
// for the odd tail
template <bool kTwBefore, bool kRealIn>
struct ColsIn {
  const void* pa;
  const void* pb;
  BigTwiddle T;
  int N2, c0, cw;
  double sgn;
  int64_t nv;  // real input: samples the signals hold (zeros beyond)
  __device__ __forceinline__ double2 operator()(int r, int c, int) const {
    double2 v = make_double2(0.0, 0.0);
    if (c < cw) {
      const int64_t idx = (int64_t)r * N2 + c0 + c;
      if (kRealIn) {
        // streaming loads (evict-first): the signal passes through once and must not push the twiddle tables out of L1
        if (idx < nv) {
          v.x = __ldcs(static_cast<const double*>(pa) + idx);
          if (pb) v.y = __ldcs(static_cast<const double*>(pb) + idx);
        }
      } else {
        v = __ldcs(static_cast<const double2*>(pa) + idx);
      }
    }
    return v;
  }
  // rows r0, r0+step, ... of column c0+c: W^(col r0) (W^(col step))^q — two table look-ups per run
  // instead of one per element (the look-ups were 2/3 of the L1 sectors of the column passes)
  template <int R>
  __device__ __forceinline__ void twiddle_run(double2 (&v)[R], int r0, int step, int c) const {
    if (!kTwBefore || c >= cw) return;
    // (measured and rejected: sincospi instead of the two look-ups each — L1TEX 63 -> 52 %, but the longer dependent
    // chain sits on the tile's critical path: 0.65 -> 0.68 ms per pass)
    double2 w = big_twiddle(T, (int64_t)r0 * (c0 + c), sgn);
    const double2 ws = big_twiddle(T, (int64_t)step * (c0 + c), sgn);
#pragma unroll
    for (int q = 0; q < R; ++q) {
      v[q] = cmul(v[q], w);
      if (q + 1 < R) w = cmul(w, ws);
    }
  }
};
template <bool kTwAfter, bool kRealOut>
struct ColsOut {
  void* pa;
  void* pb;
  BigTwiddle T;
  int N2, c0, cw;
  double sgn, scale;
  const double2* pre_w;  // compile-time path: this thread's run twiddle, fetched at kernel start (shared memory, [thread])
  int64_t nv;  // real output: samples kept (writes beyond are dropped)
  template <int R>
  __device__ __forceinline__ void twiddle_run(double2 (&v)[R], int r0, int step, int c) const {
    if (!kTwAfter || c >= cw) return;
    if (pre_w) {
      double2 w = pre_w[threadIdx.x];
      const double2 ws = pre_w[kFftColsThreads + c];
#pragma unroll
      for (int q = 0; q < R; ++q) {
        v[q] = cmul(v[q], w);
        if (q + 1 < R) w = cmul(w, ws);
      }
      return;
    }
    double2 w = big_twiddle(T, (int64_t)r0 * (c0 + c), sgn);
    const double2 ws = big_twiddle(T, (int64_t)step * (c0 + c), sgn);
#pragma unroll
    for (int q = 0; q < R; ++q) {
      v[q] = cmul(v[q], w);
      if (q + 1 < R) w = cmul(w, ws);
    }
  }
  __device__ __forceinline__ void operator()(int r, int c, int, double2 v) const {
    if (c >= cw) return;
    const int64_t idx = (int64_t)r * N2 + c0 + c;
    if (kRealOut) {
      if (idx >= nv) return;
      __stcs(static_cast<double*>(pa) + idx, v.x * scale);
      if (pb) __stcs(static_cast<double*>(pb) + idx, v.y * scale);
    } else {
      __stcs(static_cast<double2*>(pa) + idx, cscale(v, scale));
    }
  }
};
template <bool kTwAfter, bool kRealIn, bool kRealOut>
__global__ void __launch_bounds__(kFftColsThreads, kFftColsMinBlocks) fft_cols_kernel(FftPlan P, BigTwiddle T, int N2, int logc,
                                                               const void* __restrict__ in, void* __restrict__ out,
                                                               int64_t in_stride, int64_t out_stride, double sgn,
                                                               double scale, int64_t n_real, int64_t nv) {
  const int N1 = P.L, C = 1 << logc;
  double2* a = reinterpret_cast<double2*>(fft_smem_raw);
  double2* b = a + ((size_t)N1 << logc);
  const bool ct = (P.L == 625 || P.L == 640) && logc == kFftColsLogC && P.tw_in_smem && (kTwAfter ? sgn < 0.0 : sgn > 0.0);
  // (the compile-time path parks its tables behind the first stage's barrier instead of staging them in a phase of
  // their own: one barrier-bounded phase less in a tile that lives for 8 us)
  const double2* tw = ct ? P.twc : stage_twiddles(P, b + ((size_t)N1 << logc));
  const int c0 = blockIdx.x << logc;
  const int cw = min(C, N2 - c0);
  const int64_t sig = blockIdx.y;
  const bool two = 2 * sig + 1 < n_real;
  ColsIn<!kTwAfter, kRealIn> src;
  if (kRealIn) {
    src.pa = static_cast<const double*>(in) + 2 * sig * in_stride;
    src.pb = two ? static_cast<const double*>(in) + (2 * sig + 1) * in_stride : nullptr;
  } else {
    src.pa = static_cast<const double2*>(in) + sig * in_stride;
    src.pb = nullptr;
  }
  src.T = T; src.N2 = N2; src.c0 = c0; src.cw = cw; src.sgn = sgn; src.nv = nv;
  ColsOut<kTwAfter, kRealOut> dst;
  if (kRealOut) {
    dst.pa = static_cast<double*>(out) + 2 * sig * out_stride;
    dst.pb = two ? static_cast<double*>(out) + (2 * sig + 1) * out_stride : nullptr;
  } else {
    dst.pa = static_cast<double2*>(out) + sig * out_stride;
    dst.pb = nullptr;
  }
  dst.T = T; dst.N2 = N2; dst.c0 = c0; dst.cw = cw; dst.sgn = sgn; dst.scale = scale; dst.nv = nv; dst.pre_w = nullptr;
  if (ct) {
    // The filter's column passes on the grids of cfg4: 625 = 5^4 (reflection, n = 400 000) and 640 = 10 x 8 x 8 (the padded
    // kernel convolution, n = 409 600), four columns.  Every table value a thread will need is requested NOW, next to
    // the first stage's own global loads, and parked in shared memory behind that stage's barrier: the compact stage
    // twiddles and, for the pass that applies the inter-pass twiddles at its END, this thread's W^(j col) with the four
    // per-column steps W^(Ns col).  (By source line 24 % of the stall samples of these passes were first uses of such
    // look-ups, L1 misses behind the streaming signal.)
    // Thread t fetches compact twiddle t; in the last stage thread t runs butterfly t (column t % kCols, first output row
    // t / kCols, step Ns) and the last kCols threads fetch the per-column steps.
    constexpr int kCols = 1 << kFftColsLogC;
    constexpr int kTwSlot = 160;                         // compact twiddles, then kFftColsThreads + kCols run twiddles
    constexpr int kStepThread = kFftColsThreads - kCols;  // thread kStepThread + c fetches the step of column c
    static_assert(ct_twiddle_count(Radices625{}) <= kTwSlot && ct_twiddle_count(Radices640{}) <= kTwSlot, "twiddle slot");
    static_assert(kCols * ct_last_stride(Radices625{}) <= kStepThread && kCols * ct_last_stride(Radices640{}) <= kStepThread,
                  "one last-stage butterfly per thread, below the step threads");
    double2* tws = b + ((size_t)N1 << logc);
    double2* pre = tws + kTwSlot;
    const int tid = (int)threadIdx.x;
    const bool l625 = P.L == 625;
    const int n_tw = l625 ? ct_twiddle_count(Radices625{}) : ct_twiddle_count(Radices640{});
    const int ns_last = l625 ? ct_last_stride(Radices625{}) : ct_last_stride(Radices640{});
    double2 twv = make_double2(0.0, 0.0), wv = make_double2(0.0, 0.0);
    if (tid < n_tw) twv = __ldg(P.twc + tid);
    if (kTwAfter) {
      const int c = tid & (kCols - 1), j = tid >> kFftColsLogC;
      if (tid < kCols * ns_last && c < cw) wv = big_twiddle(T, (int64_t)j * (c0 + c), sgn);
      else if (tid >= kStepThread && tid - kStepThread < cw) wv = big_twiddle(T, (int64_t)ns_last * (c0 + tid - kStepThread), sgn);
      dst.pre_w = pre;
    }
    auto park = [&]() {
      if (tid < n_tw) tws[tid] = twv;
      if (kTwAfter) {
        if (tid < kCols * ns_last) pre[tid] = wv;
        else if (tid >= kStepThread) pre[kFftColsThreads + tid - kStepThread] = wv;
      }
    };
    if (l625)
      smem_fft_ct<kFftColsLogC, kTwAfter, kFftColsThreads>(Radices625{}, src, dst, tws, a, b, park);
    else
      smem_fft_ct<kFftColsLogC, kTwAfter, kFftColsThreads>(Radices640{}, src, dst, tws, a, b, park);
    return;
  }
  smem_fft(P, logc, sgn, tw, src, dst, a, b);
}

// ---- four-step, kernel B: row transforms of length N2 on scratch[k1][*] --------------
// C = 2^logc adjacent rows per CTA.
// kFilter: FFT -> * Hp[k1*N2 + k2] -> IFFT, in place (spectrum stays transposed)
// else   : FFT (sgn) and scatter to natural order out[k1 + N1*k2], scaled
struct RowsIn {
  WFM_NO_RUN_TWIDDLE
  const double2* rows;  // first row of the tile
  int N2, rw;
  __device__ __forceinline__ double2 operator()(int p, int c, int) const {
    return c < rw ? rows[(int64_t)c * N2 + p] : make_double2(0.0, 0.0);
  }
};
struct RowsOut {
  WFM_NO_RUN_TWIDDLE
  double2* rows;
  int N2, rw;
  __device__ __forceinline__ void operator()(int p, int c, int, double2 v) const {
    if (c < rw) rows[(int64_t)c * N2 + p] = v;
  }
};
struct RowsMulHOut {
  WFM_NO_RUN_TWIDDLE
  double2* z;
  const double2* __restrict__ hrows;  // Hp at the tile's first row
  int N2, rw;
  __device__ __forceinline__ void operator()(int p, int c, int e, double2 v) const {
    if (c < rw) v = cmul(v, __ldg(hrows + (int64_t)c * N2 + p));
    z[e] = v;
  }
};
struct NaturalOut {
  WFM_NO_RUN_TWIDDLE  // X[k1 + N1*k2]: for fixed k2 the C rows of the tile are adjacent
  double2* o;
  int N1, rw;
  double scale;
  __device__ __forceinline__ void operator()(int p, int c, int, double2 v) const {
    if (c < rw) o[(int64_t)c + (int64_t)N1 * p] = cscale(v, scale);
  }
};
template <bool kFilter>
__global__ void __launch_bounds__(kFftRowsThreads, kFftRowsMinBlocks) fft_rows_kernel(FftPlan P, int N1, int logc, double2* __restrict__ data,
                                                               double2* __restrict__ out, int64_t stride,
                                                               int64_t out_stride, const double2* __restrict__ Hp,
                                                               double sgn, double scale) {
  const int N2 = P.L, C = 1 << logc;
  double2* a = reinterpret_cast<double2*>(fft_smem_raw);
  double2* b = a + ((size_t)N2 << logc);
  const double2* tw = stage_twiddles(P, b + ((size_t)N2 << logc));
  const int r0 = blockIdx.x << logc;
  const int rw = min(C, N1 - r0);
  const int64_t sig = blockIdx.y;
  double2* rows = data + sig * stride + (int64_t)r0 * N2;
  if (kFilter) {
    double2* z = last_stage_target(P, a, b);
    smem_fft(P, logc, -1.0, tw, RowsIn{rows, N2, rw}, RowsMulHOut{z, Hp + (int64_t)r0 * N2, N2, rw}, a, b);
    smem_fft(P, logc, +1.0, tw, SmemIn{z}, RowsOut{rows, N2, rw}, z == a ? b : a, z);
  } else {
    smem_fft(P, logc, sgn, tw, RowsIn{rows, N2, rw}, NaturalOut{out + sig * out_stride + r0, N1, rw, scale}, a, b);
  }
}

// ---- kernel B with TMA: the tile's rows are ONE contiguous span of the scratch ---------------------------------------
// C adjacent rows of the [N1][N2] scratch are rw * N2 consecutive complex numbers, and so are the rows of the permuted
// response that multiply them.  One elected thread moves both into shared memory with cp.async.bulk (two mbarriers) and
// the filtered rows back with one bulk store: the row pass executes no LDG / STG at all — its L1TEX unit, at 76 % with
// per-thread 16-byte accesses, is left to the shared-memory traffic of the stages.  The landing buffers keep the global
// layout ([c][p]); the first stage reads it and the last one writes it through these accessors.
__device__ __forceinline__ uint32_t fft_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fft_mbar_init(uint64_t* bar) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(fft_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fft_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fft_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fft_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(fft_smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void fft_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   fft_smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(fft_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fft_bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(fft_smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
constexpr int kRowPad = 4;  // elements (64 bytes) between the rows of a landing buffer
struct RowsTileIn {
  WFM_NO_RUN_TWIDDLE
  const double2* t;  // [c][p]
  int N2;
  __device__ __forceinline__ double2 operator()(int p, int c, int) const { return t[c * N2 + p]; }
};
struct RowsTileOut {
  WFM_NO_RUN_TWIDDLE
  double2* t;  // [c][p]
  int N2;
  __device__ __forceinline__ void operator()(int p, int c, int, double2 v) const { t[c * N2 + p] = v; }
};
struct RowsTileMulHOut {
  WFM_NO_RUN_TWIDDLE
  double2* z;          // interleaved [e]
  const double2* h;    // the response rows of the tile in shared memory, [c][p]
  int N2;
  __device__ __forceinline__ void operator()(int p, int c, int e, double2 v) const { z[e] = cmul(v, h[c * N2 + p]); }
};
// dynamic shared memory of fft_rows_tma_kernel: what the row plan's buffers and table take (plan_smem, from get_plan),
// the tile's response rows, kRowPad elements behind every row of the three, and the two mbarriers
static size_t rows_tma_smem(size_t plan_smem, int L, int logc) {
  return plan_smem + sizeof(double2) * (((size_t)L << logc) + 3 * ((size_t)kRowPad << logc)) + 16;
}
__global__ void __launch_bounds__(kFftRowsThreads, kFftRowsMinBlocks) fft_rows_tma_kernel(FftPlan P, int N1, int logc,
                                                                                         double2* __restrict__ data, int64_t stride,
                                                                                         const double2* __restrict__ Hp) {
  const int N2 = P.L, C = 1 << logc;
  // landing buffers keep the global layout, one row after the other, kRowPad elements apart: with N2 a multiple of 8
  // the rows of a tile would start on the same bank group and the lanes of a butterfly pair (c = 0, 1) would collide
  const int RS = N2 + kRowPad;
  double2* a = reinterpret_cast<double2*>(fft_smem_raw);
  double2* b = a + (size_t)C * RS;  // (>= pts: the buffers also serve as the interleaved work buffers of the stages)
  double2* twp = b + (size_t)C * RS;
  double2* h = twp + P.L;
  uint64_t* bar = reinterpret_cast<uint64_t*>(h + (size_t)C * RS);
  const int r0 = blockIdx.x << logc;
  const int rw = min(C, N1 - r0);
  double2* rows = data + (int64_t)blockIdx.y * stride + (int64_t)r0 * N2;
  const uint32_t row_bytes = (uint32_t)N2 * (uint32_t)sizeof(double2);
  if (threadIdx.x == 0) {
    fft_mbar_init(bar);
    fft_mbar_init(bar + 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fft_mbar_expect_tx(bar, row_bytes * rw);
    for (int c = 0; c < rw; ++c) fft_bulk_g2s(b + (size_t)c * RS, rows + (int64_t)c * N2, row_bytes, bar);
    fft_mbar_expect_tx(bar + 1, row_bytes * rw);
    for (int c = 0; c < rw; ++c) fft_bulk_g2s(h + (size_t)c * RS, Hp + (int64_t)(r0 + c) * N2, row_bytes, bar + 1);
  }
  const bool ct = P.L == 640 && logc == kFftRowsLogC;
  const double2* tw = stage_twiddles(P, twp);  // (the launch requires the table in shared memory)
  __syncthreads();  // the barriers are initialised (and the twiddles staged) for every thread
  fft_mbar_wait(bar, 0);
  fft_mbar_wait(bar + 1, 0);
  // (a tile of fewer than C rows computes on whatever the missing rows' part of the buffers holds: columns are
  // independent and only rw rows are stored)
  double2* o = b;
  if (ct) {
    // 640 = 10 x 8 x 8, two rows: b -> a -> b -> (x H) a;  a -> b -> a -> b
    smem_fft_ct<kFftRowsLogC, true, kFftRowsThreads>(Radices640{}, RowsTileIn{b, 640 + kRowPad}, RowsTileMulHOut{a, h, 640 + kRowPad},
                                                     twp, a, b);
    smem_fft_ct<kFftRowsLogC, false, kFftRowsThreads>(Radices640{}, SmemIn{a}, RowsTileOut{b, 640 + kRowPad}, twp, b, a);
  } else {
    // (either buffer may end up holding the padded output rows: both have room for them)
    double2* z = last_stage_target(P, a, b);
    smem_fft(P, logc, -1.0, tw, RowsTileIn{b, RS}, RowsTileMulHOut{z, h, RS}, a, b);
    double2* w0 = z == a ? b : a;
    double2* oo = last_stage_target(P, w0, z);
    smem_fft(P, logc, +1.0, tw, SmemIn{z}, RowsTileOut{oo, RS}, w0, z);
    o = oo;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // this thread's tile writes -> the async proxy
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int c = 0; c < rw; ++c) fft_bulk_s2g(rows + (int64_t)c * N2, o + (size_t)c * RS, row_bytes);
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  }
}

// ---- one-level plain c2c ------------------------------------------------------------
struct PlainIn {
  WFM_NO_RUN_TWIDDLE
  const double2* d;
  __device__ __forceinline__ double2 operator()(int p, int, int) const { return d[p]; }
};
struct PlainOut {
  WFM_NO_RUN_TWIDDLE
  double2* d;
  double scale;
  __device__ __forceinline__ void operator()(int p, int, int, double2 v) const { d[p] = cscale(v, scale); }
};
__global__ void __launch_bounds__(kFftThreads) fft_c2c_single_kernel(FftPlan P, double2* __restrict__ data,
                                                                     int64_t stride, double sgn, double scale) {
  double2* a = reinterpret_cast<double2*>(fft_smem_raw);
  double2* b = a + P.L;
  const double2* tw = stage_twiddles(P, b + P.L);
  double2* d = data + (int64_t)blockIdx.x * stride;
  smem_fft(P, 0, sgn, tw, PlainIn{d}, PlainOut{d, scale}, a, b);
}

// ---- Bluestein helpers ----------------------------------------------------------------
// chirp[k] = exp(sgn * i pi k^2 / n)
__device__ __forceinline__ double2 chirp(int64_t k, int64_t n, double sgn) {
  double s, c;
  sincospi((double)((k * k) % (2 * n)) / (double)n, &s, &c);
  return make_double2(c, sgn * s);
}
// a[m] = x[m]*chirp[m] (m < n), 0 (m >= n);  per signal, length M
__global__ void bluestein_pre_kernel(const double2* __restrict__ x, int64_t x_stride, double2* __restrict__ a,
                                     int64_t n, int64_t M, double sgn) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int64_t sig = blockIdx.y;
  a[sig * M + m] = m < n ? cmul(x[sig * x_stride + m], chirp(m, n, sgn)) : make_double2(0.0, 0.0);
}
// b[m] = conj(chirp)[|m|] wrapped to length M (one copy, shared by all signals)
__global__ void bluestein_kernel_kernel(double2* __restrict__ b, int64_t n, int64_t M, double sgn) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  double2 v = make_double2(0.0, 0.0);
  if (m < n) v = chirp(m, n, -sgn);
  else if (m > M - n) v = chirp(M - m, n, -sgn);
  b[m] = v;
}
__global__ void pointwise_mul_kernel(double2* __restrict__ a, const double2* __restrict__ b, int64_t M,
                                     int64_t a_stride) {
  const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  const int64_t sig = blockIdx.y;
  a[sig * a_stride + m] = cmul(a[sig * a_stride + m], b[m]);
}
// x[k] = chirp[k] * c[k] * scale
__global__ void bluestein_post_kernel(const double2* __restrict__ c, int64_t M, double2* __restrict__ x,
                                      int64_t x_stride, int64_t n, double sgn, double scale) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t sig = blockIdx.y;
  x[sig * x_stride + k] = cscale(cmul(c[sig * M + k], chirp(k, n, sgn)), scale);
}
// pair blockIdx.y = real signals (2y, 2y+1) <-> one complex signal
__global__ void real_to_complex_kernel(const double* __restrict__ x, int64_t x_stride, double2* __restrict__ c,
                                       int64_t n, int64_t n_real) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t sig = blockIdx.y;
  const double* xa = x + 2 * sig * x_stride + k;
  c[sig * n + k] = make_double2(xa[0], 2 * sig + 1 < n_real ? xa[x_stride] : 0.0);
}
__global__ void complex_to_real_kernel(const double2* __restrict__ c, int64_t n, double* __restrict__ y,
                                       int64_t y_stride, int64_t n_real) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t sig = blockIdx.y;
  const double2 v = c[sig * n + k];
  double* ya = y + 2 * sig * y_stride + k;
  ya[0] = v.x;
  if (2 * sig + 1 < n_real) ya[y_stride] = v.y;
}

// =============================== host side =============================================
// the radix sequence of a length-n transform (distortion._fft_radices mirrors it): false if n is not 7-smooth.  The
// plan fixes the rounding of the transform, so the sequence must not change.
static bool factor_smooth(int64_t n, int* radix, int* n_stage) {
  int k = 0;
  if (n % 10 == 0) {  // a 5 takes the lone 2 the radix-8 stages would leave over
    int e = 0;
    for (int64_t m = n; m % 2 == 0; m /= 2) ++e;
    if (e % 3 == 1) {
      radix[k++] = 10;
      n /= 10;
    }
  }
  for (int r : {7, 5, 3, 8, 4, 2}) {
    while (n % r == 0) {
      if (k >= kMaxStages) return false;
      radix[k++] = r;
      n /= r;
    }
  }
  *n_stage = k;
  return n == 1;
}
static bool is_smooth(int64_t n) {
  int r[kMaxStages], k;
  return n >= 1 && factor_smooth(n, r, &k);
}

static std::mutex g_tw_mutex;
static std::map<std::pair<int, int>, double2*> g_twc_cache;             // (device, L) -> compact per-stage table
static std::map<std::pair<int, int64_t>, BigTwiddle> g_big_tw_cache;     // (device, n) -> inter-pass tables

static cudaError_t upload_table(const std::vector<double2>& host, double2** out) {
  double2* d = nullptr;
  cudaError_t e = cudaMalloc(&d, sizeof(double2) * host.size());
  if (e != cudaSuccess) return e;
  e = cudaMemcpy(d, host.data(), sizeof(double2) * host.size(), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(d); return e; }
  *out = d;
  return cudaSuccess;
}

// plan of a length-L transform run with `points` complex points per ping-pong buffer
// (L * interleave); *smem = dynamic shared memory the kernels need
static cudaError_t get_plan(int L, int64_t points, FftPlan* plan, size_t* smem) {
  plan->L = L;
  if (!factor_smooth(L, plan->radix, &plan->n_stage)) return cudaErrorInvalidValue;
  int64_t ns = 1;
  for (int s = 0; s < plan->n_stage; ++s) {
    plan->inv_ns[s] = (uint32_t)(((uint64_t(1) << 32) + ns - 1) / ns);  // exact quotient for j < 2^16
    ns *= plan->radix[s];
  }
  const size_t buffers = 2 * sizeof(double2) * (size_t)points + kPlanSlackBytes;
  plan->tw_in_smem = buffers + sizeof(double2) * (size_t)L <= (size_t)kSmemBudget;
  *smem = buffers + (plan->tw_in_smem ? sizeof(double2) * (size_t)L : 0);
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto ic = g_twc_cache.find({dev, L});
  if (ic == g_twc_cache.end()) {
    std::vector<double2> host;
    const long double two_pi = 6.283185307179586476925286766559L;
    int64_t nsc = 1;
    for (int s = 0; s < plan->n_stage; ++s) {
      for (int64_t k = 0; k < nsc; ++k) {
        // W_L^(k L / (Ns R_s)) = exp(-2 pi i k / (Ns R_s))
        long double ang = two_pi * (long double)k / (long double)(nsc * plan->radix[s]);
        host.push_back(make_double2((double)cosl(ang), (double)-sinl(ang)));
      }
      nsc *= plan->radix[s];
    }
    if (host.empty()) host.push_back(make_double2(1.0, 0.0));
    double2* d = nullptr;
    if ((e = upload_table(host, &d)) != cudaSuccess) return e;
    ic = g_twc_cache.emplace(std::make_pair(dev, L), d).first;
  }
  plan->twc = ic->second;
  plan->twc_len = 0;
  for (int64_t s2 = 0, nsc = 1; s2 < plan->n_stage; nsc *= plan->radix[s2], ++s2) plan->twc_len += (int)nsc;
  return cudaSuccess;
}

static cudaError_t get_big_twiddle(int64_t n, BigTwiddle* T) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  auto it = g_big_tw_cache.find({dev, n});
  if (it == g_big_tw_cache.end()) {
    const long double two_pi = 6.283185307179586476925286766559L;
    const int64_t n_hi = (n >> 10) + 1;
    std::vector<double2> hi((size_t)n_hi), lo(1024);
    for (int64_t h = 0; h < n_hi; ++h) {
      long double ang = two_pi * (long double)(h << 10) / (long double)n;
      hi[h] = make_double2((double)cosl(ang), (double)-sinl(ang));
    }
    for (int l = 0; l < 1024; ++l) {
      long double ang = two_pi * (long double)l / (long double)n;
      lo[l] = make_double2((double)cosl(ang), (double)-sinl(ang));
    }
    BigTwiddle t{nullptr, nullptr};
    double2 *dh = nullptr, *dl = nullptr;
    if ((e = upload_table(hi, &dh)) != cudaSuccess) return e;
    if ((e = upload_table(lo, &dl)) != cudaSuccess) { cudaFree(dh); return e; }
    t.hi = dh;
    t.lo = dl;
    it = g_big_tw_cache.emplace(std::make_pair(dev, n), t).first;
  }
  *T = it->second;
  return cudaSuccess;
}

// n = N1*N2, both 7-smooth and <= kMaxPoints, N1 as close to sqrt(n) as possible
static bool split_two_level(int64_t n, int* N1, int* N2) {
  int64_t best = 0;
  for (int64_t d = 1; d * d <= n; ++d) {
    if (n % d) continue;
    const int64_t q = n / d;
    if (q <= kMaxPoints && is_smooth(d) && is_smooth(q)) best = d;
  }
  if (!best) return false;
  *N1 = (int)best;
  *N2 = (int)(n / best);
  return true;
}

// how a length-n transform runs: one CTA per transform, four-step over the split n = N1 * N2, or (a prime factor > 7, or
// no split) through Bluestein's 7-smooth transforms
enum FftPath { kPathSingle, kPathTwoLevel, kPathGeneric };
static FftPath choose_path(int64_t n, int* N1, int* N2) {
  const bool smooth = is_smooth(n);
  if (smooth && n <= kMaxPoints) return kPathSingle;
  if (smooth && split_two_level(n, N1, N2)) return kPathTwoLevel;
  return kPathGeneric;
}

static int64_t next_smooth(int64_t m) {
  while (!is_smooth(m)) ++m;
  return m;
}

// stream-ordered scratch: keep freed blocks in the device's pool instead of returning them
// to the driver at every synchronisation (the default release threshold is 0)
static void keep_pool_memory() {
  static std::mutex mu;
  static bool done[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
  std::lock_guard<std::mutex> lock(mu);
  if (done[dev]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  done[dev] = true;
}

template <typename K>
static cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// log2 of the number of interleaved transforms per CTA: the largest power of two <= want
// whose two ping-pong buffers fit
static int tile_logc(int L, int want_log) {
  int lc = want_log;
  while (lc > 0 && ((int64_t)L << lc) > kMaxPoints) --lc;
  return lc;
}

// What the four-step transform of length n = N1 * N2 (choose_path) needs for n_tr transforms: the plans of the column
// pass (length N1) and of the row pass (length N2), the inter-pass twiddles, a scratch of n complex points per
// transform and both grids.  On success the caller owns the scratch and cudaFreeAsync's it on the stream.
struct TwoLevel {
  int lc1, lc2;  // log2 of the columns / rows per CTA
  FftPlan P1, P2;
  size_t smem1, smem2;
  BigTwiddle T;
  dim3 g1, g2;
  double2* scratch;
};
static cudaError_t two_level_setup(int64_t n, int N1, int N2, int64_t n_tr, cudaStream_t st, TwoLevel* t) {
  cudaError_t e;
  t->lc1 = tile_logc(N1, kFftColsLogC);
  t->lc2 = tile_logc(N2, kFftRowsLogC);
  if ((e = get_plan(N1, (int64_t)N1 << t->lc1, &t->P1, &t->smem1)) != cudaSuccess) return e;
  if ((e = get_plan(N2, (int64_t)N2 << t->lc2, &t->P2, &t->smem2)) != cudaSuccess) return e;
  if ((e = get_big_twiddle(n, &t->T)) != cudaSuccess) return e;
  const int C1 = 1 << t->lc1, C2 = 1 << t->lc2;
  t->g1 = dim3((unsigned)((N2 + C1 - 1) / C1), (unsigned)n_tr);
  t->g2 = dim3((unsigned)((N1 + C2 - 1) / C2), (unsigned)n_tr);
  // (Measured and rejected: running the three passes of the filter group by group of signal pairs so that a group's
  // scratch stays in the 126 MB L2 — 2.39 ms at 22 pairs per group .. 3.87 ms at 2 against 2.19 ms for one group: the
  // passes are bound on the SM (L1TEX 63-76 %, issue 43-52 %), not by HBM, and smaller grids add tails.)
  keep_pool_memory();
  t->scratch = nullptr;
  return cudaMallocAsync(&t->scratch, sizeof(double2) * (size_t)n * (size_t)n_tr, st);
}

// plain complex transform of n_sig signals, natural order, in place; n 7-smooth
static cudaError_t c2c_smooth(double2* data, int64_t n_sig, int64_t n, int64_t stride, double sgn, double scale,
                              cudaStream_t st) {
  cudaError_t e;
  int N1 = 0, N2 = 0;
  const FftPath path = choose_path(n, &N1, &N2);
  if (path == kPathSingle) {
    FftPlan P;
    size_t smem;
    if ((e = get_plan((int)n, n, &P, &smem)) != cudaSuccess) return e;
    if ((e = set_smem(fft_c2c_single_kernel, smem)) != cudaSuccess) return e;
    fft_c2c_single_kernel<<<(unsigned)n_sig, kFftThreads, smem, st>>>(P, data, stride, sgn, scale);
    return cudaGetLastError();
  }
  if (path != kPathTwoLevel) return cudaErrorNotSupported;
  TwoLevel t;
  if ((e = two_level_setup(n, N1, N2, n_sig, st, &t)) != cudaSuccess) return e;
  if ((e = set_smem(fft_cols_kernel<true, false, false>, t.smem1)) != cudaSuccess) goto done;
  fft_cols_kernel<true, false, false><<<t.g1, kFftColsThreads, t.smem1, st>>>(t.P1, t.T, N2, t.lc1, data, t.scratch, stride, n,
                                                                             sgn, 1.0, 0, n);
  if ((e = cudaGetLastError()) != cudaSuccess) goto done;
  if ((e = set_smem(fft_rows_kernel<false>, t.smem2)) != cudaSuccess) goto done;
  fft_rows_kernel<false><<<t.g2, kFftRowsThreads, t.smem2, st>>>(t.P2, N1, t.lc2, t.scratch, data, n, stride, nullptr, sgn, scale);
  e = cudaGetLastError();
done:
  cudaFreeAsync(t.scratch, st);
  return e;
}

// arbitrary n: smooth -> direct, else Bluestein
static cudaError_t c2c_any(double2* data, int64_t n_sig, int64_t n, int64_t stride, double sgn, double scale,
                           cudaStream_t st) {
  if (n <= 1) return cudaSuccess;
  int N1, N2;
  if (choose_path(n, &N1, &N2) != kPathGeneric) return c2c_smooth(data, n_sig, n, stride, sgn, scale, st);
  const int64_t M = next_smooth(2 * n - 1);
  if (choose_path(M, &N1, &N2) == kPathGeneric) return cudaErrorNotSupported;
  double2 *A = nullptr, *B = nullptr;
  cudaError_t e;
  if ((e = cudaMallocAsync(&A, sizeof(double2) * (size_t)M * (size_t)n_sig, st)) != cudaSuccess) return e;
  if ((e = cudaMallocAsync(&B, sizeof(double2) * (size_t)M, st)) != cudaSuccess) { cudaFreeAsync(A, st); return e; }
  const int T = 256;
  dim3 gM((unsigned)((M + T - 1) / T), (unsigned)n_sig), gM1((unsigned)((M + T - 1) / T), 1),
      gn((unsigned)((n + T - 1) / T), (unsigned)n_sig);
  bluestein_pre_kernel<<<gM, T, 0, st>>>(data, stride, A, n, M, sgn);
  bluestein_kernel_kernel<<<gM1, T, 0, st>>>(B, n, M, sgn);
  if ((e = c2c_smooth(A, n_sig, M, M, -1.0, 1.0, st)) != cudaSuccess) goto done;
  if ((e = c2c_smooth(B, 1, M, M, -1.0, 1.0, st)) != cudaSuccess) goto done;
  pointwise_mul_kernel<<<gM, T, 0, st>>>(A, B, M, M);
  if ((e = c2c_smooth(A, n_sig, M, M, +1.0, 1.0 / (double)M, st)) != cudaSuccess) goto done;
  bluestein_post_kernel<<<gn, T, 0, st>>>(A, M, data, stride, n, sgn, scale);
  e = cudaGetLastError();
done:
  cudaFreeAsync(A, st);
  cudaFreeAsync(B, st);
  return e;
}

// the library's status for what the transforms return: cudaErrorNotSupported stands for a length or layout they do not
// handle
static int fft_status(cudaError_t e) {
  if (e == cudaErrorNotSupported) return WFM_EUNSUPPORTED;
  return e == cudaSuccess ? WFM_OK : WFM_ECUDA;
}

}  // namespace wfm

extern "C" int wfm_fft_c2c(double* data, int64_t n_sig, int64_t n, int64_t stride, int32_t sign, void* stream) {
  using namespace wfm;
  if (!data || n_sig < 0 || n < 0 || (sign != 1 && sign != -1) || (n_sig > 1 && stride < n)) return WFM_EINVAL;
  if (n_sig == 0 || n == 0) return WFM_OK;
  const double scale = sign > 0 ? 1.0 / (double)n : 1.0;
  return fft_status(c2c_any(reinterpret_cast<double2*>(data), n_sig, n, stride, (double)sign, scale, (cudaStream_t)stream));
}

namespace wfm {

// Hermitian part of the response: Hs[k] = (H[k] + conj(H[(n-k) mod n])) / 2.  For real x,
// real(ifft(fft(x) H)) = ifft(fft(x) Hs) exactly (the anti-Hermitian part of H only feeds the
// imaginary part the reference drops with `.real`, distortion.py:210,220) — and with a
// Hermitian response TWO real signals ride through one complex transform as z = x_a + i x_b.
// H Hermitian already (reflection filters, real convolution kernels; all but the Nyquist bin):
// the sum of two equal numbers halved is exact, Hs == H bit for bit.
__device__ __forceinline__ double2 hermitian_part(const double2* __restrict__ H, int64_t k, int64_t n) {
  const double2 p = H[k], q = H[k == 0 ? 0 : n - k];
  return make_double2(0.5 * (p.x + q.x), 0.5 * (p.y - q.y));
}
__global__ void hermitian_part_kernel(const double2* __restrict__ H, double2* __restrict__ Hs, int64_t n) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) Hs[k] = hermitian_part(H, k, n);
}
// Hp[k1*N2 + k2] = Hs[k1 + N1*k2]: the transposed spectrum order the row pass produces
__global__ void permute_h_kernel(const double2* __restrict__ H, double2* __restrict__ Hp, int N1, int N2) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)N1 * N2) return;
  const int k1 = (int)(i / N2), k2 = (int)(i % N2);
  Hp[i] = hermitian_part(H, (int64_t)k1 + (int64_t)N1 * k2, (int64_t)N1 * N2);
}

// pinned staging for the caller's H (pageable host memory): the call returns without waiting
// for the stream, so the response must not be read from the caller's buffer after return.
// One buffer per calling thread; an event guards its reuse.
struct HStage {
  void* host = nullptr;
  size_t bytes = 0;
  cudaEvent_t used = nullptr;
  cudaError_t reserve(size_t need) {
    cudaError_t e = cudaSuccess;
    if (used) {
      if ((e = cudaEventSynchronize(used)) != cudaSuccess) return e;  // the previous call's copy has left the buffer
    } else if ((e = cudaEventCreateWithFlags(&used, cudaEventDisableTiming)) != cudaSuccess) {
      return e;
    }
    if (need > bytes) {
      if (host) cudaFreeHost(host);
      host = nullptr;
      bytes = 0;
      if ((e = cudaMallocHost(&host, need)) != cudaSuccess) return e;
      bytes = need;
    }
    return cudaSuccess;
  }
};
static thread_local HStage g_hstage;

}  // namespace wfm

// ---- the response in the layout the chosen path reads ---------------------------------------
// single-CTA and generic paths: the Hermitian part in natural order; two-level path: the
// Hermitian part in the transposed order the row pass produces.
namespace wfm {
// dH: natural-order response on the device -> ready (n complex, caller-allocated)
static cudaError_t prepare_response(const double2* dH, double2* ready, int64_t n, cudaStream_t st) {
  int N1 = 0, N2 = 0;
  const int T = 256;
  const unsigned gH = (unsigned)((n + T - 1) / T);
  if (choose_path(n, &N1, &N2) == kPathTwoLevel) permute_h_kernel<<<gH, T, 0, st>>>(dH, ready, N1, N2);
  else hermitian_part_kernel<<<gH, T, 0, st>>>(dH, ready, n);
  return cudaGetLastError();
}

// y = real(ifft(fft(x) * H)) with the response already prepared (prepare_response)
// n: transform length; nv <= n: samples the signals hold (the rest of the circular grid is zero padding that is never
// read or written: x and y are n_sig rows of nv samples at their pitches)
static cudaError_t run_filter(const double* x, double* y, int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                              const double2* ready, cudaStream_t st, int64_t nv = -1) {
  if (nv < 0) nv = n;
  cudaError_t e;
  int N1 = 0, N2 = 0;
  const FftPath path = choose_path(n, &N1, &N2);
  const int64_t n_pair = (n_sig + 1) / 2;  // two real signals per complex transform
  if (path == kPathSingle) {
    FftPlan P;
    size_t smem;
    if ((e = get_plan((int)n, n, &P, &smem)) != cudaSuccess) return e;
    if ((e = set_smem(fft_filter_single_kernel, smem)) != cudaSuccess) return e;
    fft_filter_single_kernel<<<(unsigned)n_pair, kFftThreads, smem, st>>>(P, x, y, x_stride, y_stride, n_sig, ready, (int)nv);
    return cudaGetLastError();
  }
  if (path == kPathTwoLevel) {
    TwoLevel t;
    if ((e = two_level_setup(n, N1, N2, n_pair, st, &t)) != cudaSuccess) return e;
    // the TMA row pass when its tile fits: the plan's table in shared memory and the response rows next to it
    const size_t smem2t = rows_tma_smem(t.smem2, N2, t.lc2);
    const bool rows_tma = t.P2.tw_in_smem && smem2t <= (size_t)kSmemBudget && t.P2.n_stage >= 1;
    if ((e = set_smem(fft_cols_kernel<true, true, false>, t.smem1)) == cudaSuccess &&
        (e = set_smem(fft_cols_kernel<false, false, true>, t.smem1)) == cudaSuccess &&
        (e = rows_tma ? set_smem(fft_rows_tma_kernel, smem2t) : set_smem(fft_rows_kernel<true>, t.smem2)) == cudaSuccess) {
      fft_cols_kernel<true, true, false><<<t.g1, kFftColsThreads, t.smem1, st>>>(t.P1, t.T, N2, t.lc1, x, t.scratch, x_stride, n,
                                                                                 -1.0, 1.0, n_sig, nv);
      if (rows_tma)
        fft_rows_tma_kernel<<<t.g2, kFftRowsThreads, smem2t, st>>>(t.P2, N1, t.lc2, t.scratch, n, ready);
      else
        fft_rows_kernel<true><<<t.g2, kFftRowsThreads, t.smem2, st>>>(t.P2, N1, t.lc2, t.scratch, nullptr, n, 0, ready, -1.0, 1.0);
      fft_cols_kernel<false, false, true><<<t.g1, kFftColsThreads, t.smem1, st>>>(t.P1, t.T, N2, t.lc1, t.scratch, y, n, y_stride,
                                                                                  +1.0, 1.0 / (double)n, n_sig, nv);
      e = cudaGetLastError();
    }
    cudaFreeAsync(t.scratch, st);
    return e;
  }
  // generic: complex copy, forward, * H, inverse, real part
  if (nv != n) return cudaErrorNotSupported;  // padded grids are chosen 7-smooth by the callers
  const int T = 256;
  const dim3 gn((unsigned)((n + T - 1) / T), (unsigned)n_pair);
  double2* c = nullptr;
  if ((e = cudaMallocAsync(&c, sizeof(double2) * (size_t)n * (size_t)n_pair, st)) != cudaSuccess) return e;
  real_to_complex_kernel<<<gn, T, 0, st>>>(x, x_stride, c, n, n_sig);
  e = c2c_any(c, n_pair, n, n, -1.0, 1.0, st);
  if (e == cudaSuccess) {
    pointwise_mul_kernel<<<gn, T, 0, st>>>(c, ready, n, n);
    e = c2c_any(c, n_pair, n, n, +1.0, 1.0 / (double)n, st);
  }
  if (e == cudaSuccess) {
    complex_to_real_kernel<<<gn, T, 0, st>>>(c, n, y, y_stride, n_sig);
    e = cudaGetLastError();
  }
  cudaFreeAsync(c, st);
  return e;
}

// H(f) = (1 - A) / (1 - A exp(-2 pi i f tau)) (distortion.py:188-205) or its reciprocal, on the np.fft.fftfreq(n, d)
// grid: f[k] = idx(k) * val, val = 1 / (n d) (numpy's own two steps), phase = ((-2 pi) f) tau rounded as numpy rounds it
__global__ void reflection_response_kernel(double2* __restrict__ H, int64_t n, double val, double A, double tau, int inverse) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t idx = k < (n + 1) / 2 ? k : k - n;
  const double f = (double)idx * val;
  const double ph = __dmul_rn(__dmul_rn(-6.283185307179586, f), tau);
  double sn, cs;
  sincos(ph, &sn, &cs);
  const double dr = 1.0 - A * cs, di = -(A * sn);  // 1 - A e
  const double g = 1.0 - A;
  if (inverse) {
    H[k] = make_double2(dr / g, di / g);
  } else {
    const double m = g / (dr * dr + di * di);
    H[k] = make_double2(dr * m, -di * m);
  }
}

// prepared responses of reflection filters, kept on the device: a flux-line calibration uses the same (A, tau) for
// every batch, the reference rebuilds H with NumPy on every call (distortion.py:209, :219)
struct ReflKey {
  int dev;
  int64_t n;
  double A, tau, fs;
  int inverse;
  bool operator==(const ReflKey& o) const {
    return dev == o.dev && n == o.n && A == o.A && tau == o.tau && fs == o.fs && inverse == o.inverse;
  }
};
struct ReflEntry {
  ReflKey key;
  double2* ready;
  cudaEvent_t done;
  uint64_t stamp;
};
static std::mutex g_refl_mu;
static std::vector<ReflEntry> g_refl_cache;
static uint64_t g_refl_clock = 0;
constexpr size_t kReflCacheEntries = 16;
}  // namespace wfm

// a response kept on the device in the layout its transform length needs (wfm_fft_response_create)
struct WfmFftResponse {
  int device;
  int64_t n;
  double2* ready;
};

extern "C" int wfm_fft_response_create(const double* H, int64_t n, WfmFftResponse** out) {
  using namespace wfm;
  if (!H || !out || n <= 0) return WFM_EINVAL;
  *out = nullptr;
  keep_pool_memory();
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return WFM_ECUDA;
  const size_t h_bytes = sizeof(double2) * (size_t)n;
  double2 *nat = nullptr, *ready = nullptr;
  const cudaStream_t st = cudaStreamPerThread;
  if (cudaMalloc(&ready, h_bytes) != cudaSuccess) return WFM_ENOMEM;
  cudaError_t e = cudaMallocAsync(&nat, h_bytes, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(nat, H, h_bytes, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = prepare_response(nat, ready, n, st);
  if (nat) cudaFreeAsync(nat, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // ready for any stream from now on
  if (e != cudaSuccess) {
    cudaFree(ready);
    return WFM_ECUDA;
  }
  *out = new WfmFftResponse{dev, n, ready};
  return WFM_OK;
}

extern "C" int wfm_fft_response_destroy(WfmFftResponse* r) {
  if (!r) return WFM_OK;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(r->device);
  cudaFree(r->ready);  // waits for work that still reads it
  if (prev >= 0) cudaSetDevice(prev);
  delete r;
  return WFM_OK;
}

extern "C" int wfm_fft_filter_prepared(const double* x, double* y, int64_t n_sig, int64_t n_valid, int64_t x_stride,
                                       int64_t y_stride, WfmFftResponse* r, void* stream) {
  using namespace wfm;
  if (!x || !y || !r || n_sig < 0 || n_valid < 0 || n_valid > r->n || (n_sig > 1 && (x_stride < n_valid || y_stride < n_valid)))
    return WFM_EINVAL;
  if (n_sig == 0 || n_valid == 0) return WFM_OK;
  keep_pool_memory();
  return fft_status(run_filter(x, y, n_sig, r->n, x_stride, y_stride, r->ready, (cudaStream_t)stream, n_valid));
}

extern "C" int wfm_fft_filter(const double* x, double* y, int64_t n_sig, int64_t n, int64_t stride, const double* H,
                              void* stream) {
  using namespace wfm;
  if (!x || !y || !H || n_sig < 0 || n < 0 || (n_sig > 1 && stride < n)) return WFM_EINVAL;
  if (n_sig == 0 || n == 0) return WFM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  keep_pool_memory();
  // H: caller's host memory -> pinned staging -> device, asynchronously
  const size_t h_bytes = sizeof(double2) * (size_t)n;
  if ((e = g_hstage.reserve(h_bytes)) != cudaSuccess) return WFM_ECUDA;
  memcpy(g_hstage.host, H, h_bytes);
  double2 *dH = nullptr, *ready = nullptr;
  if ((e = cudaMallocAsync(&dH, h_bytes, st)) != cudaSuccess) return WFM_ECUDA;
  e = cudaMemcpyAsync(dH, g_hstage.host, h_bytes, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaEventRecord(g_hstage.used, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&ready, h_bytes, st);
  if (e == cudaSuccess) e = prepare_response(dH, ready, n, st);
  int rc = e == cudaSuccess ? fft_status(run_filter(x, y, n_sig, n, stride, stride, ready, st)) : WFM_ECUDA;
  if (ready) cudaFreeAsync(ready, st);
  cudaFreeAsync(dH, st);
  return rc;
}

// reflection (inverse = 0) / correct_reflection (inverse = 1) of /root/reference/waveforms/distortion.py:208-221 for
// n_sig real signals: y = real(ifft(fft(x) * H)), resp. / H, H = reflection_filter(np.fft.fftfreq(n, 1 / sample_rate),
// A, tau) built on the device and cached.  x and y may alias; each has its own pitch.
extern "C" int wfm_reflection_filter(const double* x, double* y, int64_t n_sig, int64_t n, int64_t x_stride,
                                     int64_t y_stride, double A, double tau, double sample_rate, int32_t inverse,
                                     void* stream) {
  using namespace wfm;
  if (!x || !y || n_sig < 0 || n < 0 || (n_sig > 1 && (x_stride < n || y_stride < n)) || !(sample_rate > 0)) return WFM_EINVAL;
  if (n_sig == 0 || n == 0) return WFM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  keep_pool_memory();
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return WFM_ECUDA;
  const ReflKey key{dev, n, A, tau, sample_rate, inverse ? 1 : 0};
  double2* ready = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_refl_mu);
    for (auto& en : g_refl_cache)
      if (en.key == key) {
        en.stamp = ++g_refl_clock;
        ready = en.ready;
        if (cudaStreamWaitEvent(st, en.done, 0) != cudaSuccess) return WFM_ECUDA;  // built on another stream, maybe
        break;
      }
    if (!ready) {
      const size_t h_bytes = sizeof(double2) * (size_t)n;
      double2* nat = nullptr;
      if (g_refl_cache.size() >= kReflCacheEntries) {  // evict the least recently used response
        size_t old = 0;
        for (size_t i = 1; i < g_refl_cache.size(); ++i)
          if (g_refl_cache[i].stamp < g_refl_cache[old].stamp) old = i;
        cudaEventSynchronize(g_refl_cache[old].done);
        cudaFree(g_refl_cache[old].ready);
        cudaEventDestroy(g_refl_cache[old].done);
        g_refl_cache.erase(g_refl_cache.begin() + old);
      }
      ReflEntry en{key, nullptr, nullptr, ++g_refl_clock};
      if (cudaMalloc(&en.ready, h_bytes) != cudaSuccess) return WFM_ENOMEM;
      e = cudaMallocAsync(&nat, h_bytes, st);
      if (e == cudaSuccess) {
        const double d = 1.0 / sample_rate;            // np.fft.fftfreq(n, 1 / sample_rate): val = 1.0 / (n * d)
        const double val = 1.0 / ((double)n * d);
        reflection_response_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(nat, n, val, A, tau, inverse ? 1 : 0);
        e = cudaGetLastError();
      }
      if (e == cudaSuccess) e = prepare_response(nat, en.ready, n, st);
      if (nat) cudaFreeAsync(nat, st);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&en.done, cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventRecord(en.done, st);
      if (e != cudaSuccess) {
        cudaFree(en.ready);
        return WFM_ECUDA;
      }
      g_refl_cache.push_back(en);
      ready = en.ready;
    }
  }
  return fft_status(run_filter(x, y, n_sig, n, x_stride, y_stride, ready, st));
}
