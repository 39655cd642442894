// wfm_sample.cu — K1: batched piecewise-waveform sampling kernel for sm_100a.
//
// Replaces, for a whole batch of channels in one launch, the reference's
//   np.arange -> calc_parts (np.searchsorted, per-segment _calc/_apply,
//   np.clip) -> zeros_like -> _fill_parts
// (/root/reference/waveforms/waveform.py:173-207, :529-563, :679-693;
//  /root/reference/waveforms/_waveform.pyx:130-169).
//
// Once per program (prepare_segments_kernel / prepare_tiles_kernel / fill_packets_kernel):
//   * every segment learns the INTEGER sample position where it starts: the first
//     sample whose abscissa is >= its lower bound — a division for the guess,
//     then exact comparisons against the rounded grid value x[j] = t0 + j*delta,
//     so ownership is bit-identical to np.searchsorted on the reference's grid;
//   * every FLAT segment (no basis factor: zero, or a constant) gets its value;
//   * every ACTIVE segment gets its device program: the ABI factor rows regrouped by
//     class (sincos rows, rotation rows, generic rows; wfm_internal.h) with their
//     value slots assigned in that order, and its terms as 16-byte compact records
//     holding the byte offsets of the slots they multiply;
//   * every tile (tile_samples consecutive samples of one channel) gets ONE packet
//     with everything it needs.
//
// Per launch: a PERSISTENT grid (CTAs per SM x 148) of 8-warp CTAs in which every
// WARP is autonomous.  A warp owns a private slice of shared memory (output tile,
// value slots, two packet buffers, two mbarriers) and loops over tiles (warp w of
// the grid takes tiles w, w+G, ...); there is NO block-level barrier anywhere, so a
// warp stalled on a packet load or a long pulse never idles its neighbours.  The
// tile is ASSEMBLED IN SHARED MEMORY and leaves the SM as ONE TMA bulk store:
//   1. Prologue.  Lane 0 starts the TMA bulk load (cp.async.bulk + mbarrier) of the
//      NEXT tile's packet into the other packet buffer, then the warp waits for
//      this tile's packet (requested one tile ago).
//   2. Flat fill.  After the previous tile's bulk store has finished reading the
//      buffer, the whole tile is filled with the channel's zero-segment value
//      (16-byte shared stores, no table look-ups); the constant plateaus listed in
//      the packet are rewritten.  No abscissa is computed for flat samples.
//   3. Active samples.  The tile's active samples are grouped into UNITS (1 or 2
//      consecutive samples of one segment) that are dealt round-robin to the lanes.
//      A lane interprets the segment program once per unit — the unit's samples run
//      as independent dependency chains — and writes the values into the tile.
//   4. Store.  fence.proxy.async, __syncwarp, lane 0 issues the bulk store of the
//      whole tile with an L2 evict-first policy (the output is write-once; it must
//      not displace the IR).  HBM sees full lines only, no LSU store instructions
//      are spent on the output, and the store drains while the warp is already in
//      the prologue of its next tile.
//
// Algorithmic traffic: 8 B (4 B, 2 B) per sample, write-only.
#include <cuda_runtime.h>
#include <mutex>
#include <cstdlib>
#include <stdint.h>
#include <algorithm>
#include <type_traits>
#include "wfm_basis.cuh"
#include "wfm_multidrag.cuh"
#include "wfm_internal.h"


namespace wfm {

constexpr int kThreads = 32 * kWarps;  // autonomous warps per CTA
constexpr int kWarpsPerCta = kThreads / 32;

template <typename T> struct OutVec;
template <> struct OutVec<double> { static constexpr int N = 2; };
template <> struct OutVec<float> { static constexpr int N = 4; };
template <> struct OutVec<int16_t> { static constexpr int N = 8; };

// WFM_I16 output: 16-bit DAC codes (dac_code, wfm_math.cuh) with the gain and offset of each output row
template <typename OutT> constexpr bool kCodes = std::is_same_v<OutT, int16_t>;
// (gain, offset) of row `plane` of channel `wave` in the WfmQuant table; read where a conversion needs them, not held
// in registers across the tile loop (the sparse kernel sits at its register budget)
__device__ __forceinline__ const double* row_quant(const double* quant, int wave, int plane) {
  return quant + ((size_t)wave * 2 + plane) * 2;
}
// eight codes in one 16-byte word
__device__ __forceinline__ uint4 code_pattern(int16_t c) {
  const uint32_t w = (uint32_t)(uint16_t)c * 0x10001u;
  return make_uint4(w, w, w, w);
}

// ---- shared-memory vector stores ---------------------------------------------------
__device__ __forceinline__ void fill_vec(double* p, double v) { *reinterpret_cast<double2*>(p) = make_double2(v, v); }
__device__ __forceinline__ void fill_vec(float* p, double v) {
  const float f = (float)v;
  *reinterpret_cast<float4*>(p) = make_float4(f, f, f, f);
}
__device__ __forceinline__ void fill_vec(int16_t* p, int16_t c) { *reinterpret_cast<uint4*>(p) = code_pattern(c); }
// ---- mbarrier + TMA bulk copies ------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// size and both addresses must be multiples of 16 bytes
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global, write-once data: L2 evict-first
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  return policy;
}
__device__ __forceinline__ void bulk_s2g_evict_first(void* dst_gmem, const void* src_smem, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst_gmem),
               "r"(smem_u32(src_smem)), "r"(bytes), "l"(policy)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// generic-proxy writes to shared memory -> visible to the async proxy (TMA)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// abscissa of sample j of channel w: x[j] = t0 + j*delta — a multiply and an add,
// never fused (np.arange / np.linspace fill loops), minus the stack pre-shift.
__device__ __forceinline__ double abscissa(const WfmWave& w, const double* __restrict__ xs, int64_t j) {
  double x;
  if (w.flags & WFM_WAVE_EXPLICIT_X) {
    x = xs[w.x_off + j];
  } else {
    x = add(w.t0, mul((double)j, w.delta));
    if ((w.flags & WFM_WAVE_LAST_OVERRIDE) && j == w.n - 1) x = w.x_last;
  }
  if (w.flags & WFM_WAVE_PRESHIFT) x = sub(x, w.pre_shift);
  return x;
}

// first sample j in [0, n] of the channel with abscissa >= bound (n if none)
__device__ int first_sample_at_or_after(const WfmWave& w, const double* __restrict__ xs, int n, double bound) {
  if (!(w.flags & WFM_WAVE_EXPLICIT_X) && w.delta > 0.0) {
    double b = bound;
    if (w.flags & WFM_WAVE_PRESHIFT) b = b + w.pre_shift;
    const double g = ceil((b - w.t0) / w.delta);
    int j = g <= 0.0 ? 0 : (g >= (double)n ? n : (int)g);  // NaN -> n
    // exact fix-up against the rounded grid (monotone in j)
    while (j > 0 && abscissa(w, xs, j - 1) >= bound) --j;
    while (j < n && abscissa(w, xs, j) < bound) ++j;
    return j;
  }
  int lo = 0, hi = n;  // generic: binary search over the channel's abscissae
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (abscissa(w, xs, mid) < bound) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// the few channel fields a sample evaluation needs
struct WaveEval {
  double offset;
  uint32_t flags;
  int32_t wave;  // clip limits are read from the channel row when WFM_WAVE_CLIP is set (rare: not kept in registers)
};

// U values of one lane
template <int U>
struct Val {
  double v[U];
};
template <int U>
__device__ __forceinline__ Val<U> ld_slot(const unsigned char* p) {
  Val<U> r;
  if constexpr (U == 2) {
    const double2 d = *reinterpret_cast<const double2*>(p);
    r.v[0] = d.x;
    r.v[1] = d.y;
  } else if constexpr (U == 4) {
    // four-sample slots are two 16-byte halves 512 bytes apart (lane l at l * 16 in each): a lane-contiguous
    // 32-byte layout puts lanes l and l + 4 of a quarter warp on the same banks
    const double2 d0 = *reinterpret_cast<const double2*>(p), d1 = *reinterpret_cast<const double2*>(p + 512);
    r.v[0] = d0.x;
    r.v[1] = d0.y;
    r.v[2] = d1.x;
    r.v[3] = d1.y;
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) r.v[u] = reinterpret_cast<const double*>(p)[u];
  }
  return r;
}
template <int U>
__device__ __forceinline__ void st_slot(unsigned char* p, const Val<U>& r) {
  if constexpr (U == 2) {
    *reinterpret_cast<double2*>(p) = make_double2(r.v[0], r.v[1]);
  } else if constexpr (U == 4) {
    *reinterpret_cast<double2*>(p) = make_double2(r.v[0], r.v[1]);
    *reinterpret_cast<double2*>(p + 512) = make_double2(r.v[2], r.v[3]);
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) reinterpret_cast<double*>(p)[u] = r.v[u];
  }
}

static __device__ __noinline__ double clip_value(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// ---- the slow evaluator: ABI tables in global memory, no value cache -----------------------
// Used by cold tiles (packet larger than a buffer), wide segments (more value slots or
// terms than the hot path holds) and the complex128 kernel.  A WFM_COS_SINCOS /
// WFM_COS_ROT row IS cos(w * (x - shift)) (the lowering only regrouped equal-w cosines).
static __device__ __noinline__ double eval_row_direct(const WfmFactor& f, double x, const double* __restrict__ args) {
  if (f.func == WFM_COS_SINCOS || f.func == WFM_COS_ROT || f.func == WFM_COS) return cos_cw(mul(f.a0, sub(x, f.shift)));
  return eval_factor(FacArgs{f.func, f.arg_off, f.shift, f.a0, f.a1}, x, args);
}

// Order of operations = the reference's (_waveform.pyx:134-152, waveform.py:690-692):
// every term is amp * (((1 * f1^n1) * f2^n2) * ...), a member's terms are summed left to
// right starting from 0, the member sums are added to the accumulator (offset).
template <bool kPlanes>
static __device__ __forceinline__ void eval_segment_slow_impl(const DevProgram& P, int seg, const WaveEval& w, double x,
                                                           double& out_re, double& out_im, int plane, double offset1) {
  const WfmSegPtr p0 = P.seg_ptr[seg], p1 = P.seg_ptr[seg + 1];
  out_re = (kPlanes && plane) ? offset1 : w.offset;
  out_im = 0.0;
  if (p1.term == p0.term) return;  // zero segment: untouched by clip (calc_parts skips it)
  double g_re = 0.0, g_im = 0.0;
#pragma unroll 1
  for (int t = p0.term; t < p1.term; ++t) {
    const WfmTerm tm = P.terms[t];
    if (kPlanes && (int)((tm.flags & WFM_TERM_PLANE1) != 0) != plane) continue;
    double prod = 1.0;
#pragma unroll 1
    for (int r = 0; r < tm.n_ref; ++r) {
      const WfmRef ref = P.refs[tm.ref_begin + r];
      double v = eval_row_direct(P.facs[p0.fac + ref.slot], x, P.args);
      if (ref.kind == WFM_POW_INT) v = pow_small_int(v, (int)ref.expo);
      else if (ref.kind == WFM_POW_GEN) v = pow(v, ref.expo);
      prod = mul(prod, v);  // the reference's product starts from 1; 1 * v is exact
    }
    g_re = add(g_re, mul(tm.amp_re, prod));
    g_im = add(g_im, mul(tm.amp_im, prod));
    if (tm.flags & WFM_TERM_GROUP_END) {
      out_re = add(out_re, g_re);
      out_im = add(out_im, g_im);
      g_re = g_im = 0.0;
    }
  }
  if (w.flags & WFM_WAVE_CLIP) out_re = clip_value(out_re, P.waves[w.wave].clip_lo, P.waves[w.wave].clip_hi);
}
// (arguments and result BY VALUE: a reference would force the caller's per-sample arrays into local memory)
static __device__ __noinline__ double eval_segment_slow(const DevProgram& P, int seg, double offset, uint32_t flags, int wave,
                                                        double x) {
  double re, im;
  eval_segment_slow_impl<false>(P, seg, WaveEval{offset, flags, wave}, x, re, im, 0, 0.0);
  return re;
}
// one row of an I/Q pair: plane 0 / 1, only that row's terms are summed (row 1 starts from offset1)
static __device__ __noinline__ double eval_segment_slow_row(const DevProgram& P, int seg, double offset, uint32_t flags, int wave,
                                                            double x, int plane, double offset1) {
  double re, im;
  eval_segment_slow_impl<true>(P, seg, WaveEval{offset, flags, wave}, x, re, im, plane, offset1);
  return re;
}

// product of an extended term (more than three references or an exponent != 1) from the
// ABI tables; the factor values are the ones already sitting in the lane's value slots
static __device__ __noinline__ double term_product_ext(const DevProgram& P, int seg, int it, const unsigned char* sl, int u) {
  const int kSlotStride = slot_stride(P.unit);
  const WfmSegPtr p0 = P.seg_ptr[seg];
  const WfmTerm tm = P.terms[p0.term + it];
  double prod = 1.0;
#pragma unroll 1
  for (int r = 0; r < tm.n_ref; ++r) {
    const WfmRef ref = P.refs[tm.ref_begin + r];
    const int slot = P.row_slot[p0.fac + ref.slot];
    // sample u of the slot (four-sample units: two 16-byte halves 512 bytes apart, see ld_slot)
    const unsigned char* sp = sl + slot * kSlotStride;
    double v = P.unit == 4 ? reinterpret_cast<const double*>(sp + (u >> 1) * 512)[u & 1] : reinterpret_cast<const double*>(sp)[u];
    if (ref.kind == WFM_POW_INT) v = pow_small_int(v, (int)ref.expo);
    else if (ref.kind == WFM_POW_GEN) v = pow(v, ref.expo);
    prod = mul(prod, v);
  }
  return prod;
}

// ---- the hot evaluator: one UNIT (U samples of one active segment) per call ------------------
// blk: the segment's rows in the staged packet ({SRow CRow..}.. GRow.. CTerm..); sl: this
// lane's value slots (slot k at sl + k * kSlotStride, slot 0 holds 1.0).
// kPair: the segment may belong to an I/Q pair.  Its terms list the first row's groups, then the second row's; the
// first second-row term carries kCTermPlaneSwitch: the first row's sum is complete there, `on_switch(total)` hands it
// to the caller (who stores it) and the accumulation restarts from offset1.  `plane1` tells which row the returned
// total belongs to.
template <int U, bool kPair, typename Switch>
__device__ __forceinline__ Val<U> eval_unit(const unsigned char* __restrict__ blk, int n_sc, int n_rot, int n_gen, int n_term,
                                         const DevProgram& P, int gseg, const WaveEval& w, const double (&x)[U],
                                         unsigned char* __restrict__ sl, bool affine, const double* offset1, bool& plane1,
                                         Switch on_switch) {
  constexpr int kSlotStride = slot_stride(U);
  unsigned char* dst = sl + kSlotStride;  // slot 1
  // -- one range reduction + both polynomials per frequency; the further cosines of that
  // frequency (other shifts) by rotation of (cos, sin) while they are still in registers
  const unsigned char* __restrict__ row = blk;
#pragma unroll 1
  for (int i = 0; i < n_sc; ++i) {
    const SRow* __restrict__ sr = reinterpret_cast<const SRow*>(row);
    const double wv = sr->w;
    const int n_child = (int)sr->n_child;
    double a[U];
    Val<U> s, c;
    {
      const double shift = sr->shift;
#pragma unroll
      for (int u = 0; u < U; ++u) a[u] = mul(wv, sub(x[u], shift));
    }
    if (U >= 2 && affine) {
      // the further samples of the unit: rotation of the previous one by D = w * delta plus the MEASURED residual
      // eps = (a[u] - a[u-1]) - D (first order; |eps| ~ ulp(a)), not another range reduction
      const double a0[1] = {a[0]};
      double s0[1], c0[1];
      sincos_cw_n<1>(a0, s0, c0);
      const double D = sr->D, cD = sr->cD, sD = sr->sD;
      c.v[0] = c0[0];
      s.v[0] = s0[0];
#pragma unroll
      for (int u = 1; u < U; ++u) {
        const double eps = sub(sub(a[u], a[u - 1]), D);
        const double C = fma(c.v[u - 1], cD, -(s.v[u - 1] * sD));
        const double S = fma(s.v[u - 1], cD, c.v[u - 1] * sD);
        c.v[u] = fma(-eps, S, C);
        s.v[u] = fma(eps, C, S);
      }
    } else {
      sincos_cw_n<U>(a, s.v, c.v);
    }
    st_slot(dst, c);
    dst += kSlotStride;
    row += sizeof(SRow);
#pragma unroll 1
    for (int j = 0; j < n_child; ++j) {
      const CRow* __restrict__ cr = reinterpret_cast<const CRow*>(row);
      const double shift = cr->shift, D = cr->D, cD = cr->cD, sD = cr->sD;
      Val<U> r;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double a_t = mul(wv, sub(x[u], shift));
        // cos(a + D + eps) = C - eps S - eps^2 C / 2 ...: |eps| ~ ulp(a) (4e-11 at 1e5 rad, the
        // far end of a 100 us frame at 200 MHz), so the second-order term (< 1e-21) is dropped
        const double eps = sub(sub(a_t, a[u]), D);
        const double C = fma(c.v[u], cD, -(s.v[u] * sD));
        const double S = fma(s.v[u], cD, c.v[u] * sD);
        r.v[u] = fma(-eps, S, C);
      }
      st_slot(dst, r);
      dst += kSlotStride;
      row += sizeof(CRow);
    }
  }
  // -- every other basis function
  const GRow* __restrict__ gr = reinterpret_cast<const GRow*>(blk + n_sc * (int)sizeof(SRow) + n_rot * (int)sizeof(CRow));
#pragma unroll 1
  for (int k = 0; k < n_gen; ++k) {
    const int func = gr[k].func;
    const double shift = gr[k].shift, a0 = gr[k].a0;
    Val<U> r;
    if (func == WFM_COS) {
      double a[U], s[U];
#pragma unroll
      for (int u = 0; u < U; ++u) a[u] = mul(a0, sub(x[u], shift));
      sincos_cw_n<U>(a, s, r.v);
    } else if (func == WFM_LINEAR) {
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = sub(x[u], shift);
    } else if (func == WFM_GAUSSIAN) {
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = f_gaussian(sub(x[u], shift), a0);
    } else if (func == WFM_ERF) {
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = erf_tab(dvd(sub(x[u], shift), a0));
    } else {
      const FacArgs fa{func, gr[k].arg_off, shift, a0, gr[k].a1};
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = eval_factor(fa, x[u], P.args);
    }
    st_slot(dst, r);
    dst += kSlotStride;
  }
  // -- terms
  const uint4* __restrict__ ct = reinterpret_cast<const uint4*>(gr + n_gen);
  Val<U> total, grp;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    total.v[u] = w.offset;
    grp.v[u] = 0.0;
  }
  if constexpr (kPair) plane1 = false;
#pragma unroll 1
  for (int it = 0; it < n_term; ++it) {
    const uint4 c = ct[it];  // CTerm: amp | o0 o1 | o2 flags (offsets in bytes for THIS unit size: scaled when the packet was built)
    const double amp = __hiloint2double((int)c.y, (int)c.x);
    const uint32_t fl = c.w >> 16;
    bool ext = false;
    if (fl & (kCTermPlaneSwitch | kCTermExt)) {  // one test on the common path
      if constexpr (kPair) {
        if (fl & kCTermPlaneSwitch) {
          on_switch(total);
          plane1 = true;
#pragma unroll
          for (int u = 0; u < U; ++u) total.v[u] = *offset1;  // the packet header in shared memory: not held in registers
        }
      }
      ext = fl & kCTermExt;
    }
    Val<U> prod;
    if (ext) {
#pragma unroll
      for (int u = 0; u < U; ++u) prod.v[u] = term_product_ext(P, gseg, it, sl, u);
    } else {
      // only the references the term has (an absent one is slot 0 = 1.0: the product is the same; loading all three
      // and multiplying was measured 3.5 % slower on the dense RB batch, neutral on sparse frames)
      prod = ld_slot<U>(sl + (c.z & 0xffffu));
      if (c.z >> 16) {
        const Val<U> f1 = ld_slot<U>(sl + (c.z >> 16));
#pragma unroll
        for (int u = 0; u < U; ++u) prod.v[u] = mul(prod.v[u], f1.v[u]);
        if (c.w & 0xffffu) {
          const Val<U> f2 = ld_slot<U>(sl + (c.w & 0xffffu));
#pragma unroll
          for (int u = 0; u < U; ++u) prod.v[u] = mul(prod.v[u], f2.v[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) grp.v[u] = add(grp.v[u], mul(amp, prod.v[u]));
    if (fl & kCTermGroupEnd) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        total.v[u] = add(total.v[u], grp.v[u]);
        grp.v[u] = 0.0;
      }
    }
  }
  if (w.flags & WFM_WAVE_CLIP) {
#pragma unroll
    for (int u = 0; u < U; ++u) total.v[u] = clip_value(total.v[u], P.waves[w.wave].clip_lo, P.waves[w.wave].clip_hi);
  }
  return total;
}

// ---- the fp32 evaluator (WFM_F32 output, 1e-6 parity) --------------------------------------
// Arguments and range reductions stay in fp64 (a 200 MHz carrier reaches 1e5 rad: fp32 cannot
// even hold the argument), everything after the reduction runs in fp32: the polynomial work,
// the rotations, the products and the sums.  fp32 dependent-issue latency is a fraction of
// fp64's, which is what this kernel is bound by.  Value slots hold floats (same slot area).
template <int U>
struct ValF {
  float v[U];
};
template <int U>
__device__ __forceinline__ ValF<U> ld_slot_f(const unsigned char* p) {
  ValF<U> r;
  if constexpr (U == 2) {
    const float2 d = *reinterpret_cast<const float2*>(p);
    r.v[0] = d.x;
    r.v[1] = d.y;
  } else if constexpr (U == 4) {
    const float4 d = *reinterpret_cast<const float4*>(p);
    r.v[0] = d.x;
    r.v[1] = d.y;
    r.v[2] = d.z;
    r.v[3] = d.w;
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) r.v[u] = reinterpret_cast<const float*>(p)[u];
  }
  return r;
}
template <int U>
__device__ __forceinline__ void st_slot_f(unsigned char* p, const ValF<U>& r) {
  if constexpr (U == 2) {
    *reinterpret_cast<float2*>(p) = make_float2(r.v[0], r.v[1]);
  } else if constexpr (U == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) reinterpret_cast<float*>(p)[u] = r.v[u];
  }
}

// sin and cos of an fp64 argument to fp32 accuracy: fp64 Cody-Waite reduction (two terms of
// pi/2 are plenty for a 24-bit result), fp32 minimax kernels on [-pi/4, pi/4]
__device__ __forceinline__ void sincos_f32(double a, float& s_out, float& c_out) {
  if (!(fabs(a) <= 1073741824.0)) {
    const SinCos r = sincos_cw(a);
    s_out = (float)r.s;
    c_out = (float)r.c;
    return;
  }
  const double q = rint(a * kTrig[0]);
  double rd = fma(-q, kTrig[1], a);
  rd = fma(-q, kTrig[2], rd);
  const float r = (float)rd, z = r * r;
  // fdlibm k_sinf / k_cosf coefficients
  const float ps = fmaf(fmaf(fmaf(2.7183114939898219064e-6f, z, -1.9839334836096632576e-4f), z, 8.3333293858894631756e-3f), z,
                        -1.6666666641626524e-1f);
  const float s = fmaf(r * z, ps, r);
  const float pc = fmaf(fmaf(fmaf(2.4390448796277409065e-5f, z, -1.3886763774609929e-3f), z, 4.1666623323739063189e-2f), z,
                        -4.9999999725103100312e-1f);
  const float c = fmaf(z, pc, 1.0f);
  const int n = (int)q;
  const bool odd = n & 1;
  const float ss = odd ? c : s, cc = odd ? s : c;
  s_out = __uint_as_float(__float_as_uint(ss) ^ ((uint32_t)(n & 2) << 30));
  c_out = __uint_as_float(__float_as_uint(cc) ^ ((uint32_t)((n + 1) & 2) << 30));
}

template <int U, bool kPair, typename Switch>
__device__ __forceinline__ Val<U> eval_unit_f32(const unsigned char* __restrict__ blk, int n_sc, int n_rot, int n_gen, int n_term,
                                                const DevProgram& P, int gseg, const WaveEval& w, const double (&x)[U],
                                                unsigned char* __restrict__ sl, const double* offset1, bool& plane1,
                                                Switch on_switch) {
  constexpr int kStride = 32 * 4 * U;  // float slots: half the fp64 stride inside the same slot area
  unsigned char* dst = sl + kStride;   // slot 1 (slot 0 holds 1.0f)
  const unsigned char* __restrict__ row = blk;
#pragma unroll 1
  for (int i = 0; i < n_sc; ++i) {
    const SRow* __restrict__ sr = reinterpret_cast<const SRow*>(row);
    const double wv = sr->w, shift = sr->shift;
    const int n_child = (int)sr->n_child;
    double a[U];
    ValF<U> s, c;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      a[u] = mul(wv, sub(x[u], shift));
      sincos_f32(a[u], s.v[u], c.v[u]);
    }
    st_slot_f(dst, c);
    dst += kStride;
    row += sizeof(SRow);
#pragma unroll 1
    for (int j = 0; j < n_child; ++j) {
      const CRow* __restrict__ cr = reinterpret_cast<const CRow*>(row);
      const double cshift = cr->shift, D = cr->D;
      const float cD = (float)cr->cD, sD = (float)cr->sD;
      ValF<U> r;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float eps = (float)sub(sub(mul(wv, sub(x[u], cshift)), a[u]), D);
        const float C = fmaf(c.v[u], cD, -(s.v[u] * sD));
        const float S = fmaf(s.v[u], cD, c.v[u] * sD);
        r.v[u] = fmaf(-eps, S, C);
      }
      st_slot_f(dst, r);
      dst += kStride;
      row += sizeof(CRow);
    }
  }
  const GRow* __restrict__ gr = reinterpret_cast<const GRow*>(row);
#pragma unroll 1
  for (int k = 0; k < n_gen; ++k) {
    const int func = gr[k].func;
    const double shift = gr[k].shift, a0 = gr[k].a0;
    ValF<U> r;
    if (func == WFM_COS) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float sn;
        sincos_f32(mul(a0, sub(x[u], shift)), sn, r.v[u]);
      }
    } else if (func == WFM_LINEAR) {
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = (float)sub(x[u], shift);
    } else if (func == WFM_GAUSSIAN) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float q = (float)sub(x[u], shift) / (float)a0;
        r.v[u] = expf(-q * q);
      }
    } else if (func == WFM_ERF) {
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = erff((float)sub(x[u], shift) / (float)a0);
    } else {
      const FacArgs fa{func, gr[k].arg_off, shift, a0, gr[k].a1};
#pragma unroll
      for (int u = 0; u < U; ++u) r.v[u] = (float)eval_factor(fa, x[u], P.args);
    }
    st_slot_f(dst, r);
    dst += kStride;
  }
  const uint4* __restrict__ ct = reinterpret_cast<const uint4*>(gr + n_gen);
  ValF<U> total, grp;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    total.v[u] = (float)w.offset;
    grp.v[u] = 0.0f;
  }
  if constexpr (kPair) plane1 = false;
#pragma unroll 1
  for (int it = 0; it < n_term; ++it) {
    const uint4 c = ct[it];  // CTerm: amp | o0 o1 | o2 flags (offsets for fp64 unit-1 slots: halve for floats)
    const float amp = (float)__hiloint2double((int)c.y, (int)c.x);
    if constexpr (kPair) {
      if ((c.w >> 16) & kCTermPlaneSwitch) {
        Val<U> t0;
#pragma unroll
        for (int u = 0; u < U; ++u) t0.v[u] = (double)total.v[u];
        on_switch(t0);
        plane1 = true;
#pragma unroll
        for (int u = 0; u < U; ++u) total.v[u] = (float)*offset1;
      }
    }
    ValF<U> prod;
    if ((c.w >> 16) & kCTermExt) {
      // extended terms read fp64 slots: evaluate the segment's term in fp64 from the ABI tables
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const WfmSegPtr p0 = P.seg_ptr[gseg];
        const WfmTerm tm = P.terms[p0.term + it];
        double pr = 1.0;
        for (int r = 0; r < tm.n_ref; ++r) {
          const WfmRef ref = P.refs[tm.ref_begin + r];
          double v = (double)reinterpret_cast<const float*>(sl + P.row_slot[p0.fac + ref.slot] * kStride)[u];
          if (ref.kind == WFM_POW_INT) v = pow_small_int(v, (int)ref.expo);
          else if (ref.kind == WFM_POW_GEN) v = pow(v, ref.expo);
          pr *= v;
        }
        prod.v[u] = (float)pr;
      }
    } else {
      prod = ld_slot_f<U>(sl + ((c.z & 0xffffu) >> 1));
      if (c.z >> 16) {
        const ValF<U> f1 = ld_slot_f<U>(sl + ((c.z >> 16) >> 1));
#pragma unroll
        for (int u = 0; u < U; ++u) prod.v[u] *= f1.v[u];
        if (c.w & 0xffffu) {
          const ValF<U> f2 = ld_slot_f<U>(sl + ((c.w & 0xffffu) >> 1));
#pragma unroll
          for (int u = 0; u < U; ++u) prod.v[u] *= f2.v[u];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) grp.v[u] = fmaf(amp, prod.v[u], grp.v[u]);
    if ((c.w >> 16) & kCTermGroupEnd) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        total.v[u] += grp.v[u];
        grp.v[u] = 0.0f;
      }
    }
  }
  Val<U> out;
#pragma unroll
  for (int u = 0; u < U; ++u) out.v[u] = (double)total.v[u];
  if (w.flags & WFM_WAVE_CLIP) {
#pragma unroll
    for (int u = 0; u < U; ++u) out.v[u] = clip_value(out.v[u], P.waves[w.wave].clip_lo, P.waves[w.wave].clip_hi);
  }
  return out;
}

// ---- pre-pass (once per program) ----------------------------------------------------------
// one warp per channel: the owning channel of each of its segment rows
__global__ void mark_seg_wave_kernel(DevProgram P, int32_t* __restrict__ seg_wave, int64_t n_waves) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= n_waves) return;
  const int seg_begin = P.waves[w].seg_begin, n_seg = P.waves[w].n_seg;
  for (int k = threadIdx.x & 31; k < n_seg; k += 32) seg_wave[seg_begin + k] = (int32_t)w;
}

// samples owned by active segments (one thread per segment, after prepare_segments_kernel)
__global__ void count_active_kernel(DevProgram P, int64_t n_segs, unsigned long long* __restrict__ total) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long len = 0;
  if (s < n_segs && P.seg_ptr[s + 1].fac > P.seg_ptr[s].fac) {
    const WfmWave w = P.waves[P.seg_wave[s]];
    const int k = (int)(s - w.seg_begin);
    const int64_t hi = (k + 1 < w.n_seg) ? (int64_t)P.seg_start[s + 1] : w.n;
    len = (unsigned long long)max((int64_t)0, hi - (int64_t)P.seg_start[s]);
  }
  for (int d = 16; d; d >>= 1) len += __shfl_xor_sync(0xffffffffu, len, d);
  if ((threadIdx.x & 31) == 0 && len) atomicAdd(total, len);
}

// one thread per segment: start position, value of a flat segment, plan of an active one
__global__ void prepare_segments_kernel(DevProgram P, int32_t* __restrict__ seg_start, double* __restrict__ seg_val,
                                        double* __restrict__ seg_val1, SegPlan* __restrict__ seg_plan,
                                        uint8_t* __restrict__ row_slot, CTerm* __restrict__ cterms, int64_t n_segs) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_segs) return;
  const WfmWave w = P.waves[P.seg_wave[s]];
  const int k = (int)(s - w.seg_begin);
  seg_start[s] = k == 0 ? 0 : first_sample_at_or_after(w, P.x, (int)w.n, P.seg_bound[s - 1]);
  const WfmSegPtr p0 = P.seg_ptr[s], p1 = P.seg_ptr[s + 1];
  const int nf = p1.fac - p0.fac, nt = p1.term - p0.term;
  // value of a FLAT segment, per row of an I/Q pair: offset + sum over stack members of (0 + sum of their constant
  // terms); a row without terms here is a zero segment of that row (untouched by clip, calc_parts skips it)
  for (int plane = 0; plane < (seg_val1 ? 2 : 1); ++plane) {
    double val = plane ? w.offset2 : w.offset;
    if (nf == 0 && nt > 0) {
      double grp = 0.0;
      bool any = false;
      for (int t = p0.term; t < p1.term; ++t) {
        const WfmTerm tm = P.terms[t];
        if ((int)((tm.flags & WFM_TERM_PLANE1) != 0) != plane) continue;
        any = true;
        grp = add(grp, tm.n_ref > 0 ? CUDART_NAN : tm.amp_re);  // a term with factors would make the segment active
        if (tm.flags & WFM_TERM_GROUP_END) {
          val = add(val, grp);
          grp = 0.0;
        }
      }
      if (any && (w.flags & WFM_WAVE_CLIP)) val = fmin(fmax(val, w.clip_lo), w.clip_hi);
    }
    (plane ? seg_val1 : seg_val)[s] = val;
  }

  // plan: rows by class, value slots in class order
  int n_sc = 0, n_rot = 0, n_gen = 0;
  for (int r = 0; r < nf; ++r) {
    const int f = P.facs[p0.fac + r].func;
    if (f == WFM_COS_SINCOS) ++n_sc;
    else if (f == WFM_COS_ROT) ++n_rot;
    else if (f != WFM_NOP) ++n_gen;
  }
  const bool wide = n_sc + n_rot + n_gen > kMaxSlots || nt > 255;
  // slots: every WFM_COS_SINCOS row (ABI order) followed by the WFM_COS_ROT rows based on it, then the rest
  {
    int next = 1;
    for (int r = 0; r < nf; ++r) row_slot[p0.fac + r] = 0;
    if (!wide) {
      for (int r = 0; r < nf; ++r) {
        if (P.facs[p0.fac + r].func != WFM_COS_SINCOS) continue;
        row_slot[p0.fac + r] = (uint8_t)next++;
        for (int q = r + 1; q < nf; ++q) {
          const WfmFactor f = P.facs[p0.fac + q];
          if (f.func == WFM_COS_ROT && (int)P.args[f.arg_off] == r) row_slot[p0.fac + q] = (uint8_t)next++;
        }
      }
      for (int r = 0; r < nf; ++r) {
        const int f = P.facs[p0.fac + r].func;
        if (f != WFM_COS_SINCOS && f != WFM_COS_ROT && f != WFM_NOP) row_slot[p0.fac + r] = (uint8_t)next++;
      }
    }
  }
  for (int t = 0; t < nt; ++t) {
    const WfmTerm tm = P.terms[p0.term + t];
    bool ext = tm.n_ref > 3;
    uint16_t o[3] = {0, 0, 0};
    for (int r = 0; r < tm.n_ref && !ext; ++r) {
      const WfmRef rf = P.refs[tm.ref_begin + r];
      if (rf.kind != WFM_POW_ONE) ext = true;
      else o[r] = (uint16_t)(row_slot[p0.fac + rf.slot] * slot_stride(1));
    }
    uint16_t flags = (tm.flags & WFM_TERM_GROUP_END) ? kCTermGroupEnd : 0u;
    // the first second-row term of an I/Q pair
    if ((tm.flags & WFM_TERM_PLANE1) && (t == 0 || !(P.terms[p0.term + t - 1].flags & WFM_TERM_PLANE1))) flags |= kCTermPlaneSwitch;
    if (ext) {
      flags |= kCTermExt;
      o[0] = o[1] = o[2] = 0;
    }
    cterms[p0.term + t] = CTerm{tm.amp_re, o[0], o[1], o[2], flags};
  }
  SegPlan pl;
  pl.n_sc = (uint8_t)min(n_sc, 255);
  pl.n_rot = (uint8_t)min(n_rot, 255);
  pl.n_gen = (uint8_t)min(n_gen, 255);
  pl.flags = wide ? kSegWide : 0u;
  pl.n_term = (uint16_t)min(nt, 65535);
  pl.blk16 = wide ? 0 : (uint16_t)((n_sc * sizeof(SRow) + n_rot * sizeof(CRow) + n_gen * sizeof(GRow) + nt * sizeof(CTerm)) / 16);
  seg_plan[s] = pl;
}

// last segment k in [0, n) with start[k] <= j (start[0] == 0)
__device__ __forceinline__ int owning_segment(const int32_t* __restrict__ start, int n, int64_t j) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((int64_t)start[mid] <= j) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// what a tile's packet holds (shared by the measuring and the filling pass)
struct TileLayout {
  int n_arows, n_patch, n_units, blk16;
  bool cold;
  __device__ __forceinline__ int bytes() const {
    if (cold) return (int)sizeof(PacketHeader);
    return (int)sizeof(PacketHeader) + (n_arows ? (n_arows + 1) * (int)sizeof(ARow) : 0) + n_patch * (int)sizeof(PatchRow) +
           blk16 * 16;
  }
};

// tile-relative [a, b) of segment k (channel-relative row) clipped to the tile
__device__ __forceinline__ void seg_span(const int32_t* __restrict__ st, int n_seg, int64_t n, int k, int64_t j0, int cnt,
                                         int& a, int& b) {
  const int64_t lo = st[k], hi = (k + 1 < n_seg) ? (int64_t)st[k + 1] : n;
  a = (int)(max(lo, j0) - j0);
  b = (int)(min(hi, j0 + cnt) - j0);
}

__device__ TileLayout measure_tile(const DevProgram& P, const TileDesc& td, const WfmWave& w) {
  TileLayout L{0, 0, 0, 0, false};
  const int32_t* __restrict__ st = P.seg_start + w.seg_begin;
  const int k0 = td.seg0 - w.seg_begin;
  for (int k = k0; k < k0 + td.nb; ++k) {
    int a, b;
    seg_span(st, w.n_seg, w.n, k, td.j0, td.cnt, a, b);
    if (b <= a) continue;
    const WfmSegPtr p0 = P.seg_ptr[w.seg_begin + k], p1 = P.seg_ptr[w.seg_begin + k + 1];
    if (p1.fac > p0.fac) {
      L.n_arows += 1;
      L.blk16 += P.seg_plan[w.seg_begin + k].blk16;
      L.n_units += (b - a + P.unit - 1) / P.unit;
    } else {
      // dense programs have no base fill: every flat run is a patch row
      if (P.dense || __double_as_longlong(P.seg_val[w.seg_begin + k]) != __double_as_longlong(w.offset)) L.n_patch += 1;
      if ((w.flags & WFM_WAVE_PAIR) &&
          (P.dense || __double_as_longlong(P.seg_val1[w.seg_begin + k]) != __double_as_longlong(w.offset2)))
        L.n_patch += 1;
    }
  }
  // ARow::rel addresses 16-byte units with 12 bits
  L.cold = L.bytes() > P.pkt_cap || L.bytes() >= 4096 * 16;
  return L;
}

// the tile range t falls in: last r in [0, n_ranges) with tile_prefix[r] <= t (ranges without samples own no tile)
__device__ __forceinline__ int64_t tile_range(const int64_t* __restrict__ tile_prefix, int64_t n_ranges, int64_t t) {
  int64_t lo = 0, hi = n_ranges - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (tile_prefix[mid] <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// one thread per tile: the tile row itself (channel, sample range), the segment rows it
// spans, its packet size.  tiles / pkt_size may be NULL (sizing pass: only the statistics);
// stats[0] = largest packet (16-byte units), stats[1] = tiles whose packet does not fit.
// Tiles cover each channel from sample 0, or (windows != NULL) each window on the same grid: a window's tiles are the
// cells [k * tile_samples, (k + 1) * tile_samples) it intersects, clipped to it.  Two- and four-sample units pair the
// samples of a segment from max(segment start, tile start), so the plain program's tile grid gives the same pairs.
__global__ void prepare_tiles_kernel(DevProgram P, TileDesc* __restrict__ tiles, const int64_t* __restrict__ tile_prefix,
                                     const WfmWindow* __restrict__ windows, int64_t n_ranges, int64_t n_tiles,
                                     uint32_t* __restrict__ pkt_size, uint32_t* __restrict__ stats) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t full16 = 0, cold = 0;
  if (t < n_tiles) {
    const int64_t r = tile_range(tile_prefix, n_ranges, t);
    const int64_t wave = windows ? windows[r].wave : r;
    const WfmWave w = P.waves[wave];
    const int64_t j_begin = windows ? windows[r].j_begin : 0, j_end = windows ? windows[r].j_end : w.n;
    const int64_t out_off = windows ? windows[r].out_off : w.out_off;
    TileDesc td;
    const int64_t ts = P.tile_samples, cell = j_begin / ts + (t - tile_prefix[r]);
    td.j0 = max(j_begin, cell * ts);
    td.out0 = out_off + (td.j0 - j_begin);
    td.wave = (int32_t)wave;
    td.cnt = (int32_t)(min((cell + 1) * ts, j_end) - td.j0);
    const int32_t* st = P.seg_start + w.seg_begin;
    const int lo = owning_segment(st, w.n_seg, td.j0);
    const int hi = max(lo, owning_segment(st, w.n_seg, td.j0 + td.cnt - 1));
    td.seg0 = w.seg_begin + lo;
    td.nb = hi - lo + 1;
    TileLayout L = measure_tile(P, td, w);
    if (tiles) tiles[t] = td;
    if (pkt_size) pkt_size[t] = (uint32_t)(L.bytes() / 16);
    cold = L.cold ? 1u : 0u;
    L.cold = false;
    full16 = (uint32_t)(L.bytes() / 16);  // what the packet WOULD need
  }
  if (stats) {  // one pair of atomics per warp (every lane of the warp takes part)
    for (int d = 16; d; d >>= 1) {
      full16 = max(full16, __shfl_xor_sync(0xffffffffu, full16, d));
      cold += __shfl_xor_sync(0xffffffffu, cold, d);
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMax(stats, full16);
      if (cold) atomicAdd(stats + 1, cold);
    }
  }
}

// ---- exclusive scan of the packet sizes (three small kernels) -----------------------------
constexpr int kScanBlock = 256, kScanItems = 16, kScanTile = kScanBlock * kScanItems;  // 4096 per block

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t warp_sums[kScanBlock / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += u;
  }
  if (lane == 31) warp_sums[wid] = incl;
  __syncthreads();
  uint32_t before = 0, all = 0;
  for (int k = 0; k < kScanBlock / 32; ++k) {
    if (k < wid) before += warp_sums[k];
    all += warp_sums[k];
  }
  __syncthreads();
  *total = all;
  return before + incl - v;
}

__global__ void __launch_bounds__(kScanBlock) scan_reduce_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ sums,
                                                                 int64_t n) {
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  uint32_t v = 0;
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) v += in[base + i];
  uint32_t total;
  block_exclusive_scan(v, &total);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// single block: exclusive scan of the block sums in place; sums[n_blocks] = grand total
__global__ void __launch_bounds__(kScanBlock) scan_sums_kernel(uint32_t* __restrict__ sums, int64_t n_blocks) {
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t b0 = 0; b0 < n_blocks; b0 += kScanBlock) {
    const int64_t i = b0 + threadIdx.x;
    const uint32_t v = i < n_blocks ? sums[i] : 0;
    uint32_t total;
    const uint32_t ex = block_exclusive_scan(v, &total);
    if (i < n_blocks) sums[i] = carry + ex;
    __syncthreads();
    if (threadIdx.x == 0) carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) sums[n_blocks] = carry;
}

__global__ void __launch_bounds__(kScanBlock) scan_apply_kernel(const uint32_t* __restrict__ in, const uint32_t* __restrict__ sums,
                                                                uint32_t* __restrict__ out, int64_t n, int64_t n_blocks) {
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  uint32_t item[kScanItems];
  uint32_t v = 0;
  for (int i = 0; i < kScanItems; ++i) {
    item[i] = base + i < n ? in[base + i] : 0;
    v += item[i];
  }
  uint32_t total;
  uint32_t run = sums[blockIdx.x] + block_exclusive_scan(v, &total);
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = run;
    run += item[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = sums[n_blocks];
}

// ---- pass 2: one warp per tile writes its packet --------------------------------------------
__global__ void __launch_bounds__(256) fill_packets_kernel(DevProgram P, const TileDesc* __restrict__ tiles,
                                                           int64_t n_tiles, const WfmWindow* __restrict__ windows,
                                                           const int64_t* __restrict__ tile_prefix, int64_t n_windows,
                                                           unsigned char* __restrict__ packets) {
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= n_tiles) return;
  const TileDesc td = tiles[t];
  const WfmWave w = P.waves[td.wave];
  const TileLayout L = measure_tile(P, td, w);  // every lane, identical result
  unsigned char* pk = packets + (size_t)P.pkt_off[t] * 16;
  ARow* arows = reinterpret_cast<ARow*>(pk + sizeof(PacketHeader));
  PatchRow* patches = reinterpret_cast<PatchRow*>(arows + (L.n_arows ? L.n_arows + 1 : 0));
  unsigned char* blocks = reinterpret_cast<unsigned char*>(patches + L.n_patch);
  if (lane == 0) {
    PacketHeader h;
    h.out0 = td.out0;
    h.j0 = td.j0;
    h.base = w.offset;
    h.t0 = w.t0;
    h.delta = w.delta;
    h.wave = td.wave;
    h.flags = w.flags | (L.cold ? kPacketCold : 0u);
    h.cnt = (uint16_t)td.cnt;
    h.n_arows = L.cold ? 0 : (uint16_t)L.n_arows;
    h.n_patch = L.cold ? 0 : (uint16_t)L.n_patch;
    h.n_units = L.cold ? 0 : (uint16_t)L.n_units;
    h.reserved[0] = h.reserved[1] = 0;
    h.out1 = td.out0;
    if (w.flags & WFM_WAVE_PAIR) {  // the second row of the tile: the channel's, or its window's
      if (windows) {
        const WfmWindow win = windows[tile_range(tile_prefix, n_windows, t)];
        h.out1 = win.out_off2 + (td.j0 - win.j_begin);
      } else {
        h.out1 = w.out_off2 + td.j0;
      }
    }
    h.base1 = w.offset2;
    *reinterpret_cast<PacketHeader*>(pk) = h;
  }
  if (L.cold) return;
  // one sequential walk over the tile's segments (identical in every lane); the rows of a
  // segment are written by the lanes in parallel
  const int32_t* __restrict__ st = P.seg_start + w.seg_begin;
  const int k0 = td.seg0 - w.seg_begin;
  int ia = 0, ip = 0, first = 0;
  unsigned char* blk = blocks;
  for (int k = k0; k < k0 + td.nb; ++k) {
    int a, b;
    seg_span(st, w.n_seg, w.n, k, td.j0, td.cnt, a, b);
    if (b <= a) continue;
    const int seg = w.seg_begin + k;
    const WfmSegPtr p0 = P.seg_ptr[seg], p1 = P.seg_ptr[seg + 1];
    if (p1.fac > p0.fac) {
      const SegPlan pl = P.seg_plan[seg];
      if (lane == 0) {
        ARow r;
        r.start = (uint16_t)a;
        r.first = (uint16_t)first;
        r.rel = (uint16_t)(((blk - pk) / 16) | ((uint32_t)pl.flags << 12));
        r.len = (uint16_t)(b - a);
        r.n_sc = pl.n_sc;
        r.n_rot = pl.n_rot;
        r.n_gen = pl.n_gen;
        r.n_term = (uint8_t)pl.n_term;
        r.gseg = seg;
        arows[ia] = r;
      }
      if (!(pl.flags & kSegWide)) {
        // trig rows sit in slot order: slot s starts after (s - 1) rows, of which the SRows are 16 bytes longer
        GRow* gr = reinterpret_cast<GRow*>(blk + pl.n_sc * sizeof(SRow) + pl.n_rot * sizeof(CRow));
        CTerm* ct = reinterpret_cast<CTerm*>(gr + pl.n_gen);
        const int nf = p1.fac - p0.fac;
        for (int r = lane; r < nf; r += 32) {
          const WfmFactor f = P.facs[p0.fac + r];
          const int slot = P.row_slot[p0.fac + r];
          if (f.func == WFM_COS_SINCOS) {
            uint32_t n_child = 0;
            int g = 0;  // SRows before this one
            for (int q = 0; q < r; ++q) g += P.facs[p0.fac + q].func == WFM_COS_SINCOS;
            for (int q = r + 1; q < nf; ++q) {
              const WfmFactor c = P.facs[p0.fac + q];
              n_child += (c.func == WFM_COS_ROT && (int)P.args[c.arg_off] == r);
            }
            const double D = f.a0 * w.delta;
            double sD, cD;
            sincos(D, &sD, &cD);
            *reinterpret_cast<SRow*>(blk + (slot - 1) * sizeof(CRow) + g * (sizeof(SRow) - sizeof(CRow))) =
                SRow{f.shift, f.a0, n_child, 0u, D, cD, sD};
          } else if (f.func == WFM_COS_ROT) {
            const double* __restrict__ p = P.args + f.arg_off;  // [base_row, base_shift, D, cos D, sin D]
            int g = 0;  // SRows up to and including its parent
            for (int q = 0; q <= (int)p[0]; ++q) g += P.facs[p0.fac + q].func == WFM_COS_SINCOS;
            *reinterpret_cast<CRow*>(blk + (slot - 1) * sizeof(CRow) + g * (sizeof(SRow) - sizeof(CRow))) =
                CRow{f.shift, p[2], p[3], p[4]};
          } else if (f.func != WFM_NOP) {
            gr[slot - 1 - pl.n_sc - pl.n_rot] = GRow{f.func, f.arg_off, f.shift, f.a0, f.a1};
          }
        }
        for (int q = lane; q < p1.term - p0.term; q += 32)
          {
            // the slot offsets of the packet's terms are scaled by the unit here, once, not per evaluation
            uint4 c = reinterpret_cast<const uint4*>(P.cterms + p0.term)[q];
            const uint32_t U = (uint32_t)P.unit;
            c.z = ((c.z & 0xffffu) * U) | (((c.z >> 16) * U) << 16);
            c.w = ((c.w & 0xffffu) * U) | (c.w & 0xffff0000u);
            reinterpret_cast<uint4*>(ct)[q] = c;
          }
        blk += (size_t)pl.blk16 * 16;
      }
      ia += 1;
      first += (b - a + P.unit - 1) / P.unit;
    } else {
      const double v = P.seg_val[seg];
      if (P.dense || __double_as_longlong(v) != __double_as_longlong(w.offset)) {
        if (lane == 0) patches[ip] = PatchRow{(uint16_t)a, (uint16_t)b, 0u, v};
        ip += 1;
      }
      if (w.flags & WFM_WAVE_PAIR) {
        const double v1 = P.seg_val1[seg];
        if (P.dense || __double_as_longlong(v1) != __double_as_longlong(w.offset2)) {
          if (lane == 0) patches[ip] = PatchRow{(uint16_t)a, (uint16_t)b, 1u, v1};
          ip += 1;
        }
      }
    }
  }
  if (lane == 0 && L.n_arows) {
    ARow r{};
    r.start = (uint16_t)td.cnt;
    r.first = (uint16_t)first;
    arows[ia] = r;  // sentinel
  }
}

// ---- the sampling kernel ------------------------------------------------------------------
// [a, b) of the warp's shared tile <- val
template <typename OutT, typename T>
__device__ __forceinline__ void fill_run_value(OutT* __restrict__ s_out, int a, int b, T val, int lane) {
  constexpr int V = OutVec<OutT>::N;
  const int a_al = (a + V - 1) & ~(V - 1), b_al = b & ~(V - 1);
  if (a_al >= b_al) {
    for (int p = a + lane; p < b; p += 32) s_out[p] = (OutT)val;
    return;
  }
  if (a + lane < a_al) s_out[a + lane] = (OutT)val;
  if (b_al + lane < b) s_out[b_al + lane] = (OutT)val;
#pragma unroll 1
  for (int p = a_al + lane * V; p < b_al; p += 32 * V) fill_vec(s_out + p, val);
}
// (int16 output: the code of val with the row's (gain, offset) q)
template <typename OutT>
__device__ __forceinline__ void fill_run(OutT* __restrict__ s_out, int a, int b, double val, int lane,
                                         const double* q = nullptr) {
  if constexpr (kCodes<OutT>) fill_run_value(s_out, a, b, dac_code(val, q[0], q[1]), lane);
  else fill_run_value(s_out, a, b, val, lane);
}

// n_rows 512-byte rows of the warp's tile buffer <- val: every lane stores 16 bytes per
// row, fully unrolled per size so that the fill is n_rows stores and nothing else
template <int R>
__device__ __forceinline__ void fill_rows(unsigned char* p, uint4 v) {
#pragma unroll
  for (int r = 0; r < R; ++r) *reinterpret_cast<uint4*>(p + r * 512) = v;
}
// the 16-byte pattern of a float / double tile buffer holding val
__device__ __forceinline__ uint4 fill_pattern(double val, bool f32) {
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (__double_as_longlong(val) != 0) {
    if (f32) {
      v.x = v.y = v.z = v.w = __float_as_uint((float)val);
    } else {
      v.x = v.z = (uint32_t)__double2loint(val);
      v.y = v.w = (uint32_t)__double2hiint(val);
    }
  }
  return v;
}
__device__ __forceinline__ void fill_tile(unsigned char* p, int n_rows, uint4 v) {
  static_assert(kMaxTileSamples * 8 / 512 == 24, "the largest tile (fp64) is the first case");
  switch (n_rows) {  // tile_samples is a multiple of 128: 2 rows each in fp64, 1 row in fp32, half a row in int16
    case 24: fill_rows<24>(p, v); break;
    case 22: fill_rows<22>(p, v); break;
    case 20: fill_rows<20>(p, v); break;
    case 18: fill_rows<18>(p, v); break;
    case 16: fill_rows<16>(p, v); break;
    case 14: fill_rows<14>(p, v); break;
    case 12: fill_rows<12>(p, v); break;
    case 11: fill_rows<11>(p, v); break;
    case 10: fill_rows<10>(p, v); break;
    case 9: fill_rows<9>(p, v); break;
    case 8: fill_rows<8>(p, v); break;
    case 7: fill_rows<7>(p, v); break;
    case 6: fill_rows<6>(p, v); break;
    case 5: fill_rows<5>(p, v); break;
    case 4: fill_rows<4>(p, v); break;
    case 3: fill_rows<3>(p, v); break;
    case 2: fill_rows<2>(p, v); break;
    case 1: fill_rows<1>(p, v); break;
    default: break;
  }
}

// this lane's fp64 value slots (four-sample slots: two 16-byte halves 512 bytes apart, lane l at l * 16 in each)
template <int U>
__device__ __forceinline__ unsigned char* lane_slots(unsigned char* s_slots, int lane) {
  return s_slots + lane * (U == 4 ? 16 : 8 * U);
}

// the cold path of a tile (its packet would not fit the warp's buffers): per-sample
// search, tables in global memory, direct stores (int16 output: codes with the rows' (gain, offset) from quant)
// out1: the tile's second row (kPair: the packet header's out1, the channel's or its window's)
template <typename OutT, bool kAccumulate, bool kPair>
__device__ __forceinline__ void cold_tile(const DevProgram& P, const TileDesc& td, int64_t out1, OutT* __restrict__ out,
                                          int lane, const double* quant) {
  OutT* __restrict__ dst = out + td.out0;
  const WfmWave w = P.waves[td.wave];
  const WaveEval we{w.offset, w.flags, td.wave};
  const int32_t* __restrict__ st = P.seg_start + td.seg0;
  auto store = [&](OutT* __restrict__ row, int jj, double re, int plane) {
    if constexpr (kCodes<OutT>) {
      const double* q = row_quant(quant, td.wave, plane);
      row[jj] = dac_code(re, q[0], q[1]);
    } else {
      row[jj] = kAccumulate ? (OutT)add((double)row[jj], re) : (OutT)re;
    }
  };
  for (int jj = lane; jj < td.cnt; jj += 32) {
    int lo = 0, hi = td.nb - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((int64_t)st[mid] <= td.j0 + jj) lo = mid; else hi = mid - 1;
    }
    double re;
    const double xv = abscissa(w, P.x, td.j0 + jj);
    if (kPair && (w.flags & WFM_WAVE_PAIR)) {
      OutT* __restrict__ dst1 = out + out1;
      re = eval_segment_slow_row(P, td.seg0 + lo, we.offset, we.flags, we.wave, xv, 0, 0.0);
      store(dst, jj, re, 0);
      re = eval_segment_slow_row(P, td.seg0 + lo, we.offset, we.flags, we.wave, xv, 1, w.offset2);
      store(dst1, jj, re, 1);
    } else {
      re = eval_segment_slow(P, td.seg0 + lo, we.offset, we.flags, we.wave, xv);
      store(dst, jj, re, 0);
    }
  }
}
template <typename OutT, bool kAccumulate, bool kPair>
__device__ __noinline__ void sample_tile_cold(const DevProgram& P, const TileDesc& td, OutT* __restrict__ out, int lane) {
  cold_tile<OutT, kAccumulate, kPair>(P, td, 0, out, lane, nullptr);
}
template <bool kPair>
__device__ __noinline__ void sample_tile_cold_codes(const DevProgram& P, const TileDesc& td, int16_t* __restrict__ out,
                                                    const double* quant, int lane) {
  cold_tile<int16_t, false, kPair>(P, td, 0, out, lane, quant);
}
// I/Q pairs: the second row's position comes with the call
template <typename OutT, bool kAccumulate>
__device__ __noinline__ void sample_tile_cold_pair(const DevProgram& P, const TileDesc& td, int64_t out1,
                                                   OutT* __restrict__ out, int lane) {
  cold_tile<OutT, kAccumulate, true>(P, td, out1, out, lane, nullptr);
}
__device__ __noinline__ void sample_tile_cold_pair_codes(const DevProgram& P, const TileDesc& td, int64_t out1,
                                                         int16_t* __restrict__ out, const double* quant, int lane) {
  cold_tile<int16_t, false, true>(P, td, out1, out, lane, quant);
}

// batch size of the dynamic deal (WFM_K1_DEAL=dynamic at run time, or a large launch: dynamic_deal)
constexpr int kDealBatch = 4;
// the dense kernel's tiles are long (hundreds of active samples each): smaller batches balance the tail of a launch
constexpr int kDenseDealBatch = 2;
extern __shared__ __align__(128) unsigned char k1_smem[];

// ---- the tile pipeline of both sampling kernels ---------------------------------------------------------------------
// The warp walks its tiles and calls body(pk, flags) with every hot tile's packet in shared memory and its flags (a
// cold tile is sampled by sample_tile_cold instead); s_slots, s_pkt and s_bar are the warp's value slots, packet
// buffers and mbarriers.  Slot 0, the mbarriers, the packet double buffer and the drain of the last bulk store are
// the pipeline's.
// kBatch == 0: the static deal, warp w of the persistent grid walks tiles w, w+G, ...
// kBatch >= 2: the dynamic deal, tiles are handed out in aligned batches of kBatch consecutive tiles from a device
// counter (zeroed before the launch): warps on slower SMs simply take fewer batches.  nb = the batch this warp takes
// next; the one after is drawn one batch early by lane 0 (fetch), so nobody waits for the atomic's round trip and
// the packet pipeline can still look two tiles on
template <int kCtaWarps, int kBatch, int U, bool kF32Eval, typename OutT, bool kAccumulate, bool kPair, typename Body>
__device__ __forceinline__ void for_each_tile(const DevProgram& P, const TileDesc* tiles, int tile_begin, int tile_end,
                                              OutT* out, const double* quant, unsigned int* tile_counter,
                                              unsigned char* s_slots, unsigned char* s_pkt, uint64_t* s_bar, const Body& body) {
  static_assert(kBatch == 0 || (kBatch >= 2 && (kBatch & (kBatch - 1)) == 0), "batch: 0 or a power of two >= 2");
  const int lane = threadIdx.x & 31;
  const int n_warps = gridDim.x * kCtaWarps;
  int t, nb = 0;
  unsigned int fetch = 0;
  if constexpr (kBatch > 0) {
    unsigned int b0 = 0;
    if (lane == 0) b0 = atomicAdd(tile_counter, 2u * kBatch);  // two batches at once: the current and the next
    t = tile_begin + (int)__shfl_sync(0xffffffffu, b0, 0);
    nb = t + kBatch;
    if (lane == 0) fetch = atomicAdd(tile_counter, (unsigned int)kBatch);
  } else {
    t = tile_begin + blockIdx.x * kCtaWarps + (threadIdx.x >> 5);
  }
  auto next1 = [&](int tt) -> int {
    if constexpr (kBatch > 0) return (((tt) - tile_begin) & (kBatch - 1)) < kBatch - 1 ? tt + 1 : nb;
    else return tt + n_warps;
  };
  auto next2 = [&](int tt) -> int {
    if constexpr (kBatch > 0) {
      const int pos = (tt - tile_begin) & (kBatch - 1);
      return pos < kBatch - 2 ? tt + 2 : (pos == kBatch - 2 ? nb : nb + 1);
    } else {
      return tt + 2 * n_warps;
    }
  };
  if (t >= tile_end) return;

  if (lane == 0) {
    mbar_init(s_bar, 1);
    mbar_init(s_bar + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // slot 0: the unit a missing term reference multiplies by (the fp32 evaluator keeps float slots)
  if constexpr (kF32Eval) {
    ValF<U> one;
#pragma unroll
    for (int u = 0; u < U; ++u) one.v[u] = 1.0f;
    st_slot_f(s_slots + lane * 4 * U, one);
  } else {
    Val<U> one;
#pragma unroll
    for (int u = 0; u < U; ++u) one.v[u] = 1.0;
    st_slot(lane_slots<U>(s_slots, lane), one);
  }
  __syncwarp();

  // packet pipeline: tile t's packet is in flight into buffer 0, tile t+G's offsets sit in
  // registers (its packet goes into the other buffer at the top of iteration t).  The sparse kernel
  // sits exactly at its 128-register budget: a third pipeline stage (L2 prefetch of tile
  // t+2G) or a hoisted L2 policy register spill in this loop and cost 4-9 % (measured)
  uint32_t off_next = 0, end_next = 0;  // packet of tile t + G, 16-byte units
  {
    const uint32_t o0 = P.pkt_off[t], o1 = P.pkt_off[t + 1];
    if (lane == 0) {
      mbar_expect_tx(s_bar, (o1 - o0) * 16u);
      bulk_g2s(s_pkt, P.packets + (size_t)o0 * 16, (o1 - o0) * 16u, s_bar);
    }
    if (next1(t) < tile_end) {
      off_next = P.pkt_off[next1(t)];
      end_next = P.pkt_off[next1(t) + 1];
    }
  }
  // it = tiles this warp has started: packet buffer it & 1, whose mbarrier completes its (it >> 1)-th phase
  uint32_t it = 0;
  auto advance = [&]() {
    if constexpr (kBatch > 0) {
      // leaving the last tile of a batch: this warp moves into batch nb and draws the one after the next
      const bool last = ((t - tile_begin) & (kBatch - 1)) == kBatch - 1;
      t = next1(t);
      if (last) {
        nb = tile_begin + (int)__shfl_sync(0xffffffffu, fetch, 0);
        if (lane == 0) fetch = atomicAdd(tile_counter, (unsigned int)kBatch);
      }
    } else {
      t += n_warps;
    }
  };
#pragma unroll 1
  for (; t < tile_end; advance()) {
    const int buf = (int)(it & 1u);
    const unsigned char* pk = s_pkt + (size_t)buf * P.pkt_cap;
    // prefetch: the next tile's packet into the other buffer (its previous tile is done:
    // every lane passed the __syncwarp that ends an iteration), the offsets of the tile after.
    // (Per-lane cp.async instead of the bulk copy was measured 5 % slower.)
    if (next1(t) < tile_end) {
      if (lane == 0) {
        mbar_expect_tx(s_bar + (buf ^ 1), (end_next - off_next) * 16u);
        bulk_g2s(s_pkt + (size_t)(buf ^ 1) * P.pkt_cap, P.packets + (size_t)off_next * 16, (end_next - off_next) * 16u,
                 s_bar + (buf ^ 1));
      }
      if (next2(t) < tile_end) {
        off_next = P.pkt_off[next2(t)];
        end_next = P.pkt_off[next2(t) + 1];
      }
    }
    mbar_wait(s_bar + buf, (it >> 1) & 1u);

    // (the cold tile ends its iteration on its own: one shared tail for both paths costs the sparse kernel 4-16 bytes
    // of spills at its 128-register budget, ptxas -v)
    const uint32_t flags = reinterpret_cast<const PacketHeader*>(pk)->flags;
    if (flags & kPacketCold) {
      if constexpr (kPair) {
        const int64_t out1 = reinterpret_cast<const PacketHeader*>(pk)->out1;
        if constexpr (kCodes<OutT>) sample_tile_cold_pair_codes(P, tiles[t], out1, out, quant, lane);
        else sample_tile_cold_pair<OutT, kAccumulate>(P, tiles[t], out1, out, lane);
      } else {
        if constexpr (kCodes<OutT>) sample_tile_cold_codes<kPair>(P, tiles[t], out, quant, lane);
        else sample_tile_cold<OutT, kAccumulate, kPair>(P, tiles[t], out, lane);
      }
      __syncwarp();
      ++it;
      continue;
    }
    body(pk, flags);
    __syncwarp();  // all reads of the packet are done: its buffer may be refilled
    ++it;
  }
  if (lane == 0) bulk_wait_read_all();  // shared memory must outlive the reads of a tile's bulk store
}

// ---- the active samples of a tile, shared by both sampling kernels -------------------------------------------------
// The tile's units are dealt round-robin to the lanes.  Per unit: its abscissae, the evaluator (the slow one for a wide
// segment, else the fp32 or the fp64 interpreter) and, in an I/Q pair, the switch to the second row.  The results go
// to sink(plane1, jj, n_valid, r): samples jj .. jj + n_valid - 1 of the tile in row plane1 of the pair.
// s_slots: the warp's value slots, sl: this lane's (lane_slots).
template <int U, bool kPair, bool kF32Eval, typename Sink>
__device__ __forceinline__ void eval_units(const DevProgram& P, const unsigned char* pk, double base,
                                           uint32_t flags, int cnt, int n_units, unsigned char* s_slots, unsigned char* sl,
                                           int lane, const Sink& sink) {
  if (n_units <= 0) return;
  const PacketHeader* __restrict__ h = reinterpret_cast<const PacketHeader*>(pk);
  const ARow* __restrict__ arows = reinterpret_cast<const ARow*>(pk + sizeof(PacketHeader));
  const WaveEval we{base, flags, h->wave};
  const double t0 = h->t0, delta = h->delta;
  const int64_t j0 = h->j0;
  const bool plain_grid = !(flags & (WFM_WAVE_EXPLICIT_X | WFM_WAVE_LAST_OVERRIDE | WFM_WAVE_PRESHIFT));
  int lo = 0;
#pragma unroll 1
  for (int i = lane; i < n_units; i += 32) {
    while ((int)arows[lo + 1].first <= i) ++lo;  // the active segment holding unit i (i grows monotonically)
    const uint4 rw = reinterpret_cast<const uint4*>(arows)[lo];  // ARow: start first | rel len | n_sc n_rot n_gen n_term | gseg
    const int start = rw.x & 0xffffu, first = rw.x >> 16, rel = rw.y & 0xfffu, len = rw.y >> 16;
    const uint32_t sflags = (rw.y >> 12) & 0xfu;
    const int jj = start + (i - first) * U;
    const int n_valid = min(U, start + len - jj);
    double x[U];
    if (plain_grid) {
      // the tile's sample index fits 32 bits (channels hold < 2^31 samples)
      const int jg = (int)j0 + jj;
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = add(t0, mul((double)(jg + u), delta));
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = abscissa(P.waves[h->wave], P.x, j0 + min(jj + u, cnt - 1));
    }
    Val<U> r;
    bool plane1 = false;
    // the first row of an I/Q pair is complete when its last term has been added
    auto first_row = [&](const Val<U>& v) { sink(false, jj, n_valid, v); };
    if (sflags & kSegWide) {
      if constexpr (kPair) {
#pragma unroll
        for (int u = 0; u < U; ++u) r.v[u] = eval_segment_slow_row(P, (int)rw.w, we.offset, we.flags, we.wave, x[u], 0, 0.0);
        if (flags & WFM_WAVE_PAIR) {
          first_row(r);
          plane1 = true;
#pragma unroll
          for (int u = 0; u < U; ++u) r.v[u] = eval_segment_slow_row(P, (int)rw.w, we.offset, we.flags, we.wave, x[u], 1, h->base1);
        }
      } else {
#pragma unroll
        for (int u = 0; u < U; ++u) r.v[u] = eval_segment_slow(P, (int)rw.w, we.offset, we.flags, we.wave, x[u]);
      }
    } else if constexpr (kF32Eval) {
      r = eval_unit_f32<U, kPair>(pk + rel * 16, rw.z & 0xffu, (rw.z >> 8) & 0xffu, (rw.z >> 16) & 0xffu, rw.z >> 24, P,
                                  (int)rw.w, we, x, s_slots + lane * 4 * U, &h->base1, plane1, first_row);
    } else {
      r = eval_unit<U, kPair>(pk + rel * 16, rw.z & 0xffu, (rw.z >> 8) & 0xffu, (rw.z >> 16) & 0xffu, rw.z >> 24, P,
                              (int)rw.w, we, x, sl, !(flags & WFM_WAVE_EXPLICIT_X), &h->base1, plane1, first_row);
    }
    sink(plane1, jj, n_valid, r);
  }
}

// kF32Eval (float output only): the fp32 EVALUATOR (eval_unit_f32) instead of the fp64 one rounded at the store.
// Faster, but its error is ~1e-7 x (sum of the term magnitudes), so segments whose terms cancel (a DRAG scaling with
// w * s >> 1) leave the 1e-6 tolerance: WFM_F32_FAST is opt-in, WFM_F32 always evaluates in fp64.
template <typename OutT, bool kAccumulate, int U, int kBatch, bool kPair, bool kF32Eval>
__global__ void __launch_bounds__(kThreads, kMinBlocks)
    sample_kernel(const __grid_constant__ DevProgram P, const TileDesc* __restrict__ tiles, int tile_begin, int tile_end,
                  OutT* __restrict__ out, unsigned int* __restrict__ tile_counter, const double* __restrict__ quant) {
  constexpr int V = OutVec<OutT>::N;
  // an accumulating launch keeps its tile buffer in fp64, so that the epilogue adds the fp64 value to out and rounds
  // once (an fp32 buffer would round twice); packet_capacity sizes every program's slice for fp64 tile buffers
  using TileT = std::conditional_t<kAccumulate, double, OutT>;
  const int lane = threadIdx.x & 31;
  // this warp's private slice
  const WarpSlice ws = warp_slice(kPair ? 2 : 1, P.tile_samples, sizeof(TileT), P.n_slots, U, P.pkt_cap);
  unsigned char* slice = k1_smem + (size_t)(threadIdx.x >> 5) * ws.bytes();
  TileT* s_out = reinterpret_cast<TileT*>(slice);
  unsigned char* s_slots = slice + ws.slots();
  unsigned char* sl = lane_slots<U>(s_slots, lane);

  // a unit's results -> the tile buffer of its row
  auto to_tile = [&](bool plane1, int jj, int n_valid, const Val<U>& r) {
    TileT* row_buf = plane1 ? s_out + P.tile_samples : s_out;
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (u < n_valid) row_buf[jj + u] = (TileT)r.v[u];
  };
  for_each_tile<kWarpsPerCta, kBatch, U, kF32Eval, OutT, kAccumulate, kPair>(
      P, tiles, tile_begin, tile_end, out, quant, tile_counter, s_slots, slice + ws.packets(),
      reinterpret_cast<uint64_t*>(slice + ws.barriers()), [&](const unsigned char* pk, uint32_t flags) {
        const PacketHeader* __restrict__ h = reinterpret_cast<const PacketHeader*>(pk);
        const int cnt = h->cnt;
        const int n_arows = h->n_arows, n_patch = h->n_patch, n_units = h->n_units;
        const double base = h->base;
        OutT* __restrict__ dst = out + h->out0;

        // the previous tile's bulk store must have finished READING the tile buffer
        if (lane == 0) bulk_wait_read_all();  // returns at once when no store is outstanding
        __syncwarp();

        // base fill: the whole tile BUFFER (tile_samples, a multiple of 128) <- the zero-segment
        // value; flat segments with another value and the active samples overwrite it below
        const int tile_bytes = P.tile_samples * (int)sizeof(TileT);
        auto base_fill = [&](TileT* buf, double val, int plane) {
          unsigned char* p = reinterpret_cast<unsigned char*>(buf) + lane * 16;
          if constexpr (kCodes<OutT>) {
            const double* q = row_quant(quant, h->wave, plane);
            const uint4 v = code_pattern(dac_code(val, q[0], q[1]));
            fill_tile(p, tile_bytes / 512, v);
            // an odd multiple of 128 samples ends in half a 512-byte row
            if ((tile_bytes & 511) && lane < 16) *reinterpret_cast<uint4*>(p + (tile_bytes & ~511)) = v;
          } else {
            fill_tile(p, tile_bytes / 512, fill_pattern(val, sizeof(TileT) == 4));
          }
        };
        base_fill(s_out, base, 0);
        if constexpr (kPair) {
          if (flags & WFM_WAVE_PAIR) base_fill(s_out + P.tile_samples, h->base1, 1);
        }
        __syncwarp();

        const ARow* __restrict__ arows = reinterpret_cast<const ARow*>(pk + sizeof(PacketHeader));
        const PatchRow* __restrict__ patches = reinterpret_cast<const PatchRow*>(arows + (n_arows ? n_arows + 1 : 0));
        // ---- flat segments with their own value ----------------------------------------------
        for (int i = 0; i < n_patch; ++i) {
          if constexpr (kCodes<OutT>) {
            const int plane = kPair && patches[i].plane;
            fill_run(plane ? s_out + P.tile_samples : s_out, (int)patches[i].a, (int)patches[i].b, patches[i].val, lane,
                     row_quant(quant, h->wave, plane));
          } else {
            fill_run(kPair && patches[i].plane ? s_out + P.tile_samples : s_out, (int)patches[i].a, (int)patches[i].b,
                     patches[i].val, lane);
          }
        }

        // ---- the tile's ACTIVE samples ---------------------------------------------------------
        if constexpr (kCodes<OutT>) {
          // a unit's codes -> the tile buffer of its row
          eval_units<U, kPair, kF32Eval>(P, pk, base, flags, cnt, n_units, s_slots, sl, lane,
                                         [&](bool plane1, int jj, int n_valid, const Val<U>& r) {
                                           const double* q = row_quant(quant, h->wave, plane1);
                                           OutT* row_buf = plane1 ? s_out + P.tile_samples : s_out;
#pragma unroll
                                           for (int u = 0; u < U; ++u)
                                             if (u < n_valid) row_buf[jj + u] = dac_code(r.v[u], q[0], q[1]);
                                         });
        } else {
          eval_units<U, kPair, kF32Eval>(P, pk, base, flags, cnt, n_units, s_slots, sl, lane, to_tile);
        }

        // ---- store ---------------------------------------------------------------------------
        if (kAccumulate) {
          // out += tile (WfmLaunch::accumulate): read-modify-write epilogue, one rounding to OutT
          __syncwarp();
          for (int p = lane; p < cnt; p += 32) dst[p] = (OutT)add((double)dst[p], (double)s_out[p]);
          if constexpr (kPair) {
            if (flags & WFM_WAVE_PAIR) {
              OutT* __restrict__ dst1 = out + h->out1;
              for (int p = lane; p < cnt; p += 32) dst1[p] = (OutT)add((double)dst1[p], (double)s_out[P.tile_samples + p]);
            }
          }
        } else {
          // the whole tile as one TMA bulk copy (an I/Q pair: one per row)
          fence_proxy_async_smem();
          __syncwarp();
          const int n_bulk = cnt & ~(V - 1);  // 16-byte multiple (8 codes, 4 floats, 2 doubles); the ragged tail goes out as scalars
          if (lane == 0 && n_bulk > 0) {
            const uint64_t policy = l2_evict_first_policy();
            bulk_s2g_evict_first(dst, s_out, (uint32_t)n_bulk * sizeof(OutT), policy);
            if constexpr (kPair) {
              if (flags & WFM_WAVE_PAIR)
                bulk_s2g_evict_first(out + h->out1, s_out + P.tile_samples, (uint32_t)n_bulk * sizeof(OutT), policy);
            }
          }
          if (n_bulk + lane < cnt) {
            dst[n_bulk + lane] = s_out[n_bulk + lane];
            if constexpr (kPair) {
              if (flags & WFM_WAVE_PAIR) (out + h->out1)[n_bulk + lane] = s_out[P.tile_samples + n_bulk + lane];
            }
          }
        }
      });
}

// ---- the DENSE sampling kernel -------------------------------------------------------------
// Programs whose samples are mostly ACTIVE (randomized-benchmarking batches: back-to-back pulses) are bound by the
// interpreter, not by the store: ncu on cfg3 showed 28 % of the issued instructions were fp64 arithmetic, the rest
// row / term decoding, slot traffic and the unit bookkeeping, all paid once per UNIT.  This kernel therefore
//   * evaluates FOUR consecutive samples per lane unit (the decode cost per sample halves against two; samples 1..3
//     take their (cos, sin) from the previous one by rotation: one range reduction per frequency and unit),
//   * runs ONE CTA of 12 autonomous warps per SM at up to 168 registers (the four dependency chains of a unit are
//     the latency hiding that the second CTA used to provide),
//   * stores results straight from registers (two 16-byte stores per lane and row; a warp round covers 1 KB of
//     consecutive samples) — no tile buffer, so a warp's shared-memory slice holds only value slots and packets and
//     the tile can be long,
//   * writes flat runs (zero / constant segments, ALL listed as patch rows in dense programs) directly as well.
// Packets, the pre-pass, the deal of the tiles and the evaluator are the sparse kernel's.
constexpr int kDenseThreads = 32 * kDenseWarps;

// U consecutive results -> global memory (16-byte stores when the address allows; int16 output: the codes with the
// row's (gain, offset) q, one 8-byte store)
template <typename OutT, bool kAccumulate, int U>
__device__ __forceinline__ void store_unit(OutT* __restrict__ p, const Val<U>& r, int n_valid, const double* q = nullptr) {
  if constexpr (kCodes<OutT>) {
    static_assert(U == 4 && !kAccumulate, "int16 dense stores are one short4, never accumulated");
    int16_t c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) c[u] = dac_code(r.v[u], q[0], q[1]);
    if (n_valid == U && ((uintptr_t)p & 7) == 0) {
      *reinterpret_cast<short4*>(p) = make_short4(c[0], c[1], c[2], c[3]);
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (u < n_valid) p[u] = c[u];
    }
    return;
  }
  if (kAccumulate) {
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (u < n_valid) p[u] = (OutT)add((double)p[u], r.v[u]);
    return;
  }
  if (n_valid == U && ((uintptr_t)p & 15) == 0) {
    if constexpr (sizeof(OutT) == 8) {
#pragma unroll
      for (int u = 0; u < U; u += 2) *reinterpret_cast<double2*>(p + u) = make_double2(r.v[u], r.v[u + 1]);
    } else {
      static_assert(U == 4, "fp32 dense stores are one float4");
      *reinterpret_cast<float4*>(p) = make_float4((float)r.v[0], (float)r.v[1], (float)r.v[2], (float)r.v[3]);
    }
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (u < n_valid) p[u] = (OutT)r.v[u];
  }
}

// [a, b) of a channel row <- val, by the whole warp (int16 output: its code with the row's (gain, offset) q)
template <typename OutT, bool kAccumulate>
__device__ __forceinline__ void fill_global(OutT* __restrict__ row, int a, int b, double val, int lane,
                                            const double* q = nullptr) {
  if constexpr (kCodes<OutT>) {
    static_assert(!kAccumulate, "codes are never accumulated");
    const int16_t c = dac_code(val, q[0], q[1]);
    const int mis = (int)(((uintptr_t)(row + a) & 15) / sizeof(OutT));
    const int head = min(b - a, mis ? 8 - mis : 0);
    if (lane < head) row[a + lane] = c;
    const int a2 = a + head, nvec = (b - a2) / 8;
    const uint4 v = code_pattern(c);
    for (int k = lane; k < nvec; k += 32) *reinterpret_cast<uint4*>(row + a2 + k * 8) = v;
    const int t0 = a2 + nvec * 8;
    if (t0 + lane < b) row[t0 + lane] = c;
    return;
  }
  if (kAccumulate) {
    if (val != 0.0)
      for (int p = a + lane; p < b; p += 32) row[p] = (OutT)add((double)row[p], val);
    return;
  }
  constexpr int V = OutVec<OutT>::N;
  // head up to the first 16-byte boundary, vector body, tail
  const int mis = (int)(((uintptr_t)(row + a) & 15) / sizeof(OutT));
  const int head = min(b - a, mis ? V - mis : 0);
  if (lane < head) row[a + lane] = (OutT)val;
  const int a2 = a + head, nvec = (b - a2) / V;
  for (int q = lane; q < nvec; q += 32) {
    if constexpr (sizeof(OutT) == 8) *reinterpret_cast<double2*>(row + a2 + q * V) = make_double2(val, val);
    else {
      const float f = (float)val;
      *reinterpret_cast<float4*>(row + a2 + q * V) = make_float4(f, f, f, f);
    }
  }
  const int t0 = a2 + nvec * V;
  if (t0 + lane < b) row[t0 + lane] = (OutT)val;
}

template <typename OutT, bool kAccumulate, int kBatch, bool kPair, bool kF32Eval>
__global__ void __launch_bounds__(kDenseThreads, 1)
    sample_dense_kernel(const __grid_constant__ DevProgram P, const TileDesc* __restrict__ tiles, int tile_begin, int tile_end,
                        OutT* __restrict__ out, unsigned int* __restrict__ tile_counter, const double* __restrict__ quant) {
  constexpr int U = kDenseUnit;
  const int lane = threadIdx.x & 31;
  const WarpSlice ws = warp_slice(0, 0, 0, P.n_slots, U, P.pkt_cap);
  unsigned char* slice = k1_smem + (size_t)(threadIdx.x >> 5) * ws.bytes();
  unsigned char* s_slots = slice + ws.slots();
  unsigned char* sl = lane_slots<U>(s_slots, lane);
  for_each_tile<kDenseWarps, kBatch, U, kF32Eval, OutT, kAccumulate, kPair>(
      P, tiles, tile_begin, tile_end, out, quant, tile_counter, s_slots, slice + ws.packets(),
      reinterpret_cast<uint64_t*>(slice + ws.barriers()), [&](const unsigned char* pk, uint32_t flags) {
        const PacketHeader* __restrict__ h = reinterpret_cast<const PacketHeader*>(pk);
        const int n_arows = h->n_arows, n_patch = h->n_patch, n_units = h->n_units;
        OutT* __restrict__ dst0 = out + h->out0;
        OutT* dst1 = dst0;
        if constexpr (kPair) dst1 = out + h->out1;
        const ARow* __restrict__ arows = reinterpret_cast<const ARow*>(pk + sizeof(PacketHeader));
        const PatchRow* __restrict__ patches = reinterpret_cast<const PatchRow*>(arows + (n_arows ? n_arows + 1 : 0));
        // ---- flat runs: every zero / constant segment of the tile is listed (dense programs) --------------------------
        for (int i = 0; i < n_patch; ++i) {
          if constexpr (kCodes<OutT>) {
            const int plane = kPair && patches[i].plane;
            fill_global<OutT, false>(plane ? dst1 : dst0, (int)patches[i].a, (int)patches[i].b, patches[i].val, lane,
                                     row_quant(quant, h->wave, plane));
          } else {
            fill_global<OutT, kAccumulate>((kPair && patches[i].plane) ? dst1 : dst0, (int)patches[i].a, (int)patches[i].b,
                                           patches[i].val, lane);
          }
        }
        // ---- active samples: units of four, results straight to global memory ----------------------------------------
        eval_units<U, kPair, kF32Eval>(P, pk, h->base, flags, h->cnt, n_units, s_slots, sl, lane,
                                       [&](bool plane1, int jj, int n_valid, const Val<U>& r) {
                                         if constexpr (kCodes<OutT>)
                                           store_unit<OutT, false, U>((plane1 ? dst1 : dst0) + jj, r, n_valid,
                                                                      row_quant(quant, h->wave, plane1));
                                         else
                                           store_unit<OutT, kAccumulate, U>((plane1 ? dst1 : dst0) + jj, r, n_valid);
                                       });
      });
}

// complex128 output: the real and the imaginary PLANE are sampled by the real-valued kernel
// (a planar twin of the program, wfm_api.cu) into scratch; this kernel interleaves them
// tile by tile (exactly the samples of the requested channels, no padding touched), both
// rows of an I/Q pair (blockIdx.y = row).  im == nullptr: a real program read as complex.
template <bool kAccumulate>
__global__ void __launch_bounds__(256) interleave_c128_kernel(const TileDesc* __restrict__ tiles, const WfmWave* __restrict__ waves,
                                                              const double* __restrict__ re, const double* __restrict__ im,
                                                              double2* __restrict__ out) {
  const TileDesc td = tiles[blockIdx.x];
  int64_t off = td.out0;
  if (blockIdx.y) {
    const WfmWave& w = waves[td.wave];
    if (!(w.flags & WFM_WAVE_PAIR)) return;
    off = w.out_off2 + td.j0;
  }
  const double* __restrict__ r = re + off;
  const double* __restrict__ i = im ? im + off : nullptr;
  double2* __restrict__ dst = out + off;
  for (int j = threadIdx.x; j < td.cnt; j += blockDim.x) {
    double2 v = make_double2(r[j], i ? i[j] : 0.0);
    if (kAccumulate) {
      const double2 o = dst[j];
      v.x = add(o.x, v.x);
      v.y = add(o.y, v.y);
    }
    dst[j] = v;
  }
}

cudaError_t launch_interleave_c128(const TileDesc* tiles, int64_t n_tiles, const WfmWave* waves, bool pairs, const double* re,
                                   const double* im, void* out, int accumulate, cudaStream_t stream) {
  if (n_tiles == 0) return cudaSuccess;
  const dim3 grid((unsigned)n_tiles, pairs ? 2 : 1);
  if (accumulate) interleave_c128_kernel<true><<<grid, 256, 0, stream>>>(tiles, waves, re, im, (double2*)out);
  else interleave_c128_kernel<false><<<grid, 256, 0, stream>>>(tiles, waves, re, im, (double2*)out);
  return cudaGetLastError();
}

cudaError_t launch_prepare_segments(const DevProgram& P, const PrepareCounts& n, const PrepareBuffers& b, cudaStream_t stream) {
  const int threads = 128;
  auto blocks = [&](int64_t items) { return (unsigned)((items + threads - 1) / threads); };
  if (n.n_waves > 0 && n.n_segs > 0) mark_seg_wave_kernel<<<blocks(n.n_waves * 32), threads, 0, stream>>>(P, b.seg_wave, n.n_waves);
  if (n.n_segs > 0)
    prepare_segments_kernel<<<blocks(n.n_segs), threads, 0, stream>>>(P, b.seg_start, b.seg_val, b.seg_val1, b.seg_plan,
                                                                      b.row_slot, b.cterms, n.n_segs);
  return cudaGetLastError();
}

cudaError_t launch_count_active(const DevProgram& P, int64_t n_segs, unsigned long long* total, cudaStream_t stream) {
  if (n_segs <= 0) return cudaSuccess;
  count_active_kernel<<<(unsigned)((n_segs + 127) / 128), 128, 0, stream>>>(P, n_segs, total);
  return cudaGetLastError();
}

cudaError_t launch_prepare_tiles(const DevProgram& P, const PrepareCounts& n, const PrepareBuffers& b, uint32_t* stats,
                                 cudaStream_t stream) {
  if (n.n_tiles <= 0) return cudaSuccess;
  const int threads = 128;
  prepare_tiles_kernel<<<(unsigned)((n.n_tiles + threads - 1) / threads), threads, 0, stream>>>(
      P, b.tiles, b.tile_prefix, b.windows, b.windows ? n.n_windows : n.n_waves, n.n_tiles, b.pkt_size, stats);
  return cudaGetLastError();
}

// one block: the whole scan of a small program in one launch (the README example has 16 tiles)
__global__ void __launch_bounds__(kScanBlock) scan_small_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int n) {
  const int base = threadIdx.x * kScanItems;
  uint32_t item[kScanItems];
  uint32_t v = 0;
  for (int i = 0; i < kScanItems; ++i) {
    item[i] = base + i < n ? in[base + i] : 0;
    v += item[i];
  }
  uint32_t total;
  uint32_t run = block_exclusive_scan(v, &total);
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = run;
    run += item[i];
  }
  if (threadIdx.x == 0) out[n] = total;
}

cudaError_t launch_scan(const uint32_t* pkt_size, uint32_t* pkt_off, uint32_t* scratch, int64_t n, cudaStream_t stream) {
  const int64_t n_blocks = (n + kScanTile - 1) / kScanTile;
  if (n_blocks == 0) return cudaMemsetAsync(pkt_off, 0, sizeof(uint32_t), stream);
  if (n_blocks == 1) {
    scan_small_kernel<<<1, kScanBlock, 0, stream>>>(pkt_size, pkt_off, (int)n);
    return cudaGetLastError();
  }
  scan_reduce_kernel<<<(unsigned)n_blocks, kScanBlock, 0, stream>>>(pkt_size, scratch, n);
  scan_sums_kernel<<<1, kScanBlock, 0, stream>>>(scratch, n_blocks);
  scan_apply_kernel<<<(unsigned)n_blocks, kScanBlock, 0, stream>>>(pkt_size, scratch, pkt_off, n, n_blocks);
  return cudaGetLastError();
}

cudaError_t launch_fill_packets(const DevProgram& P, const TileDesc* tiles, int64_t n_tiles, const PrepareCounts& n,
                                const PrepareBuffers& b, unsigned char* packets, cudaStream_t stream) {
  if (n_tiles == 0) return cudaSuccess;
  fill_packets_kernel<<<(unsigned)((n_tiles + 7) / 8), 256, 0, stream>>>(P, tiles, n_tiles, b.windows, b.tile_prefix,
                                                                         n.n_windows, packets);
  return cudaGetLastError();
}

size_t sample_smem_bytes(const DevProgram& P, int dtype, bool accumulate) {
  const int elem = dtype == WFM_F32 && !accumulate ? 4 : (dtype == WFM_I16 ? 2 : 8);
  return (size_t)(P.dense ? kDenseWarps : kWarpsPerCta) * program_slice(P, P.tile_samples, elem, P.pkt_cap).bytes();
}

// tile counters of the dynamic deal: one ring per device, never freed
constexpr int kCounterSlots = 1024;
struct CounterRing {
  unsigned int* counters = nullptr;
  cudaEvent_t used[kCounterSlots] = {};
  int next = 0;
  std::mutex mu;
};
static CounterRing* counter_ring(int dev) {
  static std::mutex mu;
  static CounterRing* rings[64] = {};
  if (dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lk(mu);
  if (!rings[dev]) {
    CounterRing* r = new CounterRing;
    if (cudaMalloc(&r->counters, sizeof(unsigned int) * kCounterSlots) != cudaSuccess) {
      delete r;
      return nullptr;
    }
    rings[dev] = r;
  }
  return rings[dev];
}

// Per kernel instantiation and device: the shared-memory attribute and the occupancy of the (few) slice sizes seen so
// far, so that a steady-state launch costs one cudaGetDevice and the launch itself (the README example spends more
// time in cudaFuncSetAttribute / cudaOccupancyMax... than in the kernel).
struct LaunchCfg {
  int sms = 0;
  size_t smem_attr = 0;  // largest dynamic shared-memory size the attribute has been raised to
  struct Occ {
    size_t smem;
    int per_sm;
  };
  Occ occ[8] = {};
  int n_occ = 0;
};
template <typename K>
static cudaError_t launch_cfg(K k, LaunchCfg* table, std::mutex& mu, size_t smem, int* sms, int* per_sm, int threads = kThreads) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
  std::lock_guard<std::mutex> lk(mu);
  LaunchCfg& c = table[dev];
  if (!c.sms && (e = cudaDeviceGetAttribute(&c.sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  if (smem > c.smem_attr) {
    if ((e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    c.smem_attr = smem;
  }
  *sms = c.sms;
  for (int i = 0; i < c.n_occ; ++i)
    if (c.occ[i].smem == smem) {
      *per_sm = c.occ[i].per_sm;
      return cudaSuccess;
    }
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k, threads, smem)) != cudaSuccess) return e;
  c.occ[c.n_occ % 8] = LaunchCfg::Occ{smem, *per_sm};
  c.n_occ = std::min(c.n_occ + 1, 8);
  return cudaSuccess;
}

// One launch of a sampling kernel: the persistent grid (every warp walks tiles w, w+G, ... or draws batches of kBatch
// tiles), at most one warp per tile.  The shared-memory attribute and occupancy table is per kernel instantiation.
template <auto kKernel, int kThreadsPerCta, int kBatch, typename OutT>
static cudaError_t launch_kernel(const DevProgram& P, const TileDesc* tiles, int64_t tile_begin, int64_t n_tiles, int dtype,
                                 bool accumulate, void* out, const double* quant, cudaStream_t stream) {
  static LaunchCfg cfg_table[64];
  static std::mutex cfg_mu;
  const int warps = kThreadsPerCta / 32;
  const size_t smem = sample_smem_bytes(P, dtype, accumulate);
  int dev = 0, sms = 0, per_sm = 0;
  cudaError_t e = launch_cfg(kKernel, cfg_table, cfg_mu, smem, &sms, &per_sm, kThreadsPerCta);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorInvalidConfiguration;
  const unsigned grid = (unsigned)std::min<int64_t>((n_tiles + warps - 1) / warps, (int64_t)sms * per_sm);
  if (kBatch == 0) {
    kKernel<<<grid, kThreadsPerCta, smem, stream>>>(P, tiles, (int)tile_begin, (int)(tile_begin + n_tiles), (OutT*)out, nullptr,
                                                    quant);
    return cudaGetLastError();
  }
  // the tile counter of this launch: the next slot of a per-device ring (allocated once), zeroed on the launch's
  // stream; the slot's event makes a launch that comes kCounterSlots launches later wait for this one.  The ring's
  // mutex is held until the event is recorded: a thread that wraps around to this slot waits for THIS launch.
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  CounterRing* ring = counter_ring(dev);
  if (!ring) return cudaErrorMemoryAllocation;
  std::lock_guard<std::mutex> lk(ring->mu);
  const int slot = ring->next;
  ring->next = (ring->next + 1) % kCounterSlots;
  if (!ring->used[slot]) {
    if ((e = cudaEventCreateWithFlags(&ring->used[slot], cudaEventDisableTiming)) != cudaSuccess) return e;
  } else if ((e = cudaStreamWaitEvent(stream, ring->used[slot], 0)) != cudaSuccess) {
    return e;
  }
  unsigned int* counter = ring->counters + slot;
  if ((e = cudaMemsetAsync(counter, 0, sizeof(unsigned int), stream)) != cudaSuccess) return e;
  kKernel<<<grid, kThreadsPerCta, smem, stream>>>(P, tiles, (int)tile_begin, (int)(tile_begin + n_tiles), (OutT*)out, counter,
                                                  quant);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return cudaEventRecord(ring->used[slot], stream);
}

// The deal of a launch.  Dynamic (batches of tiles drawn from a counter) is the default whenever the warps have several
// batches each to draw: measured +7..10 % on near-pure-store programs (cfg4) and on very uneven tiles (cfg5), +2 % on
// dense cfg3, +-1 % on the control frames (cfg2), DESIGN.md; small launches keep the static deal (no counter to allocate
// and zero).  Sparse: >= ~7 tiles per warp of a full persistent grid, fp64 output only (fp32 tiles are half as long,
// the counter traffic doubles: 856 static against 811-822 GSa/s dynamic on cfg2).  Dense: >= 8192 tiles.
// WFM_K1_DEAL=static|dynamic overrides, for every launch.
static bool dynamic_deal(const DevProgram& P, int64_t n_tiles, int dtype) {
  const char* dv = getenv("WFM_K1_DEAL");  // a scan of environ (~0.1 us); read per launch so that tests can flip it
  const char deal = dv ? dv[0] : '\0';
  if (deal == 'd') return true;
  if (deal == 's') return false;
  return P.dense ? n_tiles >= (int64_t)8 * 1024 : n_tiles >= (int64_t)16 * 1024 && dtype == WFM_F64;
}

// f(std::true_type) or f(std::false_type): a run-time flag as a compile-time one
template <typename F>
static cudaError_t with_bool(bool b, F&& f) {
  return b ? f(std::true_type{}) : f(std::false_type{});
}

// the kernel for one output type: dense or sparse (unit 1 / 2), I/Q pairs or not, static or dynamic deal
template <typename OutT, bool kAcc, bool kFast>
static cudaError_t launch_typed(const DevProgram& P, const TileDesc* tiles, int64_t tile_begin, int64_t n_tiles, int dtype,
                                bool dynamic, void* out, const double* quant, cudaStream_t stream) {
  return with_bool(P.planes == 2, [&](auto pair) {
    return with_bool(dynamic, [&](auto dyn) {
      constexpr bool kPair = decltype(pair)::value;
      if (P.dense) {
        constexpr int kBatch = decltype(dyn)::value ? kDenseDealBatch : 0;
        return launch_kernel<sample_dense_kernel<OutT, kAcc, kBatch, kPair, kFast>, kDenseThreads, kBatch, OutT>(
            P, tiles, tile_begin, n_tiles, dtype, kAcc, out, quant, stream);
      }
      constexpr int kBatch = decltype(dyn)::value ? kDealBatch : 0;
      return with_bool(P.unit == 2, [&](auto u2) {
        constexpr int U = decltype(u2)::value ? 2 : 1;
        return launch_kernel<sample_kernel<OutT, kAcc, U, kBatch, kPair, kFast>, kThreads, kBatch, OutT>(
            P, tiles, tile_begin, n_tiles, dtype, kAcc, out, quant, stream);
      });
    });
  });
}

cudaError_t launch_sample(const DevProgram& P, const TileDesc* tiles, int64_t tile_begin, int64_t n_tiles, int dtype,
                          int accumulate, void* out, cudaStream_t stream, const double* quant) {
  if (n_tiles == 0) return cudaSuccess;
  if (tile_begin + n_tiles > INT32_MAX) return cudaErrorInvalidValue;
  // WFM_I16: codes from the fp64 evaluator, never accumulated
  if (dtype == WFM_I16) {
    if (accumulate || !quant) return cudaErrorInvalidValue;
    return launch_typed<int16_t, false, false>(P, tiles, tile_begin, n_tiles, dtype, dynamic_deal(P, n_tiles, dtype), out,
                                               quant, stream);
  }
  // WFM_F32_FAST: float output by the fp32 evaluator (not with accumulate: that is the careful path anyway)
  const bool fast32 = dtype == WFM_F32_FAST && !accumulate;
  if (dtype == WFM_F32_FAST) dtype = WFM_F32;
  if (dtype != WFM_F64 && dtype != WFM_F32) return cudaErrorInvalidValue;  // WFM_C128 is assembled from two real planes (wfm_api.cu)
  const bool dynamic = dynamic_deal(P, n_tiles, dtype);
  return with_bool(fast32, [&](auto fast) {
    return with_bool(dtype == WFM_F64 && !fast32, [&](auto f64) {
      return with_bool(accumulate && !fast32, [&](auto acc) {
        constexpr bool kFast = decltype(fast)::value, kAcc = decltype(acc)::value;
        using OutT = std::conditional_t<decltype(f64)::value, double, float>;
        if constexpr (kFast && (sizeof(OutT) == 8 || kAcc)) {
          return cudaErrorInvalidValue;  // not reached: the fp32 evaluator writes float and never accumulates
        } else {
          return launch_typed<OutT, kAcc, kFast>(P, tiles, tile_begin, n_tiles, dtype, dynamic, out, nullptr, stream);
        }
      });
    });
  });
}

// ---- wfm_quantize: f64 rows -> 16-bit DAC codes -----------------------------------------------------------------
// One thread per 8 consecutive samples of a row: four 16-byte loads and one 16-byte store when both rows allow it
// (kVec), scalar accesses otherwise.  Grid: x over the row, y over the rows.
constexpr int kQuantThreads = 256;
template <bool kVec>
__global__ void __launch_bounds__(kQuantThreads) quantize_kernel(const double* __restrict__ x, int16_t* __restrict__ y,
                                                                  int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                                                                  const double* __restrict__ gain_offset) {
  const int64_t j = ((int64_t)blockIdx.x * kQuantThreads + threadIdx.x) * 8;
  if (j >= n) return;
  for (int64_t s = blockIdx.y; s < n_sig; s += gridDim.y) {
    const double g = gain_offset[2 * s], o = gain_offset[2 * s + 1];
    const double* __restrict__ xr = x + s * x_stride + j;
    int16_t* __restrict__ yr = y + s * y_stride + j;
    if (kVec && j + 8 <= n) {
      int16_t c[8];
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        const double2 v = __ldcs(reinterpret_cast<const double2*>(xr + k));
        c[k] = dac_code(v.x, g, o);
        c[k + 1] = dac_code(v.y, g, o);
      }
      uint4 w;
      w.x = (uint32_t)(uint16_t)c[0] | ((uint32_t)(uint16_t)c[1] << 16);
      w.y = (uint32_t)(uint16_t)c[2] | ((uint32_t)(uint16_t)c[3] << 16);
      w.z = (uint32_t)(uint16_t)c[4] | ((uint32_t)(uint16_t)c[5] << 16);
      w.w = (uint32_t)(uint16_t)c[6] | ((uint32_t)(uint16_t)c[7] << 16);
      *reinterpret_cast<uint4*>(yr) = w;
    } else {
      for (int k = 0; k < 8 && j + k < n; ++k) yr[k] = dac_code(xr[k], g, o);
    }
  }
}

cudaError_t launch_quantize(const double* x, int16_t* y, int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                            const double* gain_offset, cudaStream_t stream) {
  if (n_sig <= 0 || n <= 0) return cudaSuccess;
  const bool vec = ((uintptr_t)x % 16) == 0 && ((uintptr_t)y % 16) == 0 && (x_stride % 2) == 0 && (y_stride % 8) == 0;
  const dim3 grid((unsigned)((n + 8 * kQuantThreads - 1) / (8 * kQuantThreads)), (unsigned)std::min<int64_t>(n_sig, 65535));
  if (vec) quantize_kernel<true><<<grid, kQuantThreads, 0, stream>>>(x, y, n_sig, n, x_stride, y_stride, gain_offset);
  else quantize_kernel<false><<<grid, kQuantThreads, 0, stream>>>(x, y, n_sig, n, x_stride, y_stride, gain_offset);
  return cudaGetLastError();
}

}  // namespace wfm
