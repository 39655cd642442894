/*
 * wfm_b200.h — C-ABI of the B200 waveform sampling engine (libwfmb200.so).
 *
 * The reference (feihoo87/waveforms 2.2.3) has no FFI for this path: the seam
 * is Python-level.  Each entry point below names the reference call it
 * replaces (paths relative to /root/reference):
 *
 *   wfm_program_create   – the walk over (bounds, seq) that
 *                          waveforms/_waveform.pyx:155-169 (calc_parts) does
 *                          per call; here the piecewise program is uploaded
 *                          once as a flat IR and reused.
 *   wfm_program_create_windows
 *                        – Waveform.__call__(x, frag=True) batched: a program
 *                          that samples and stores only given windows of its
 *                          channels (the non-zero runs), packed.
 *   wfm_sample           – Waveform.sample / Waveform.__call__ /
 *                          WaveVStack.__call__  (waveforms/waveform.py:173-207,
 *                          :529-563, :679-693) = np.arange + calc_parts +
 *                          _calc/_apply + basis functions
 *                          (_waveform.pyx:130-152, :290-371;
 *                          multy_drag.py:158-232) + np.clip + _fill_parts.
 *   wfm_sample_host      – same, with HOST output buffers (device->host copy
 *                          inside the call): the end-to-end path.
 *   wfm_sample_quant(_host), wfm_quantize
 *                        – no reference counterpart: 16-bit DAC codes
 *                          (gain, offset, round, saturate) converted in the
 *                          kernel's store instead of NumPy on the host.
 *   wfm_sosfilt          – scipy.signal.sosfilt call sites
 *                          waveforms/waveform.py:200-203, :249.
 *   wfm_lfilter,
 *   wfm_lfilter_mode     – scipy.signal.lfilter in distortion.py:321 (predistort):
 *                          sequential bit-identical kernel, or block-parallel
 *                          scan for orders <= 4.
 *   wfm_fft_filter,
 *   wfm_reflection_filter,
 *   wfm_fft_response_create / wfm_fft_filter_prepared
 *                        – np.fft.fft / ifft in distortion.py:208-221
 *                          (reflection, correct_reflection; the response built
 *                          and cached on the device) and
 *                          scipy.signal.fftconvolve in distortion.py:329-333
 *                          (the kernel's response prepared once).
 *   wfm_expand_templates – no reference counterpart (the reference builds one
 *                          Python object per pulse, _waveform.pyx:68-88,
 *                          :216-235): per-pulse IR rows written on the device
 *                          from pulse templates + per-pulse payloads.
 *   wfm_calibrate_fp64 / wfm_calibrate_copy
 *                        – in-run FP64 and pinned-copy ceilings for bench.py.
 *
 * Conventions: plain C structs of pointers and counts; every function returns
 * 0 on success or a negative WFM_E* code (no exceptions cross the ABI), and
 * wfm_last_error() returns a thread-local message.  Device output buffers are
 * caller-owned (the library never frees them).  Calls are asynchronous with
 * respect to `stream` (a cudaStream_t passed as void*, NULL = legacy default
 * stream) unless the name ends in _host.  One program lives on one device;
 * multi-GPU callers create one program per device holding that device's shard
 * of the channels (no collective is involved anywhere on this path).
 */
#ifndef WFM_B200_H
#define WFM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WFM_ABI_VERSION 2

/* error codes */
#define WFM_OK            0
#define WFM_EINVAL       -1  /* malformed IR / bad argument            */
#define WFM_ECUDA        -2  /* CUDA runtime error (see last_error)    */
#define WFM_ENOMEM       -3
#define WFM_EUNSUPPORTED -4  /* basis id or mode not implemented       */

/* basis-function ids — identical to the reference's registration order
 * (_waveform.pyx:374-388; multy_drag.py:177, :214) */
enum {
  WFM_LINEAR = 1, WFM_GAUSSIAN = 2, WFM_ERF = 3, WFM_COS = 4, WFM_SINC = 5,
  WFM_EXP = 6, WFM_INTERP = 7, WFM_LINEARCHIRP = 8, WFM_EXPONENTIALCHIRP = 9,
  WFM_HYPERBOLICCHIRP = 10, WFM_COSH = 11, WFM_SINH = 12, WFM_DRAG = 13,
  WFM_MOLLIFIER = 14, WFM_D_GAUSSIAN = 15, WFM_DRAG_SIN = 16,
  WFM_DRAG_SINX = 17,
  /* lowering-only ops (never appear in Waveform objects); DESIGN.md, K1:
   * several COS factors of one segment that share w are evaluated as ONE sincos
   * plus rotations by the exactly measured argument difference */
  WFM_COS_SINCOS = 32, /* slot k <- cos(w(x-shift)), slot k+1 <- sin(...); the
                          next factor row must be WFM_NOP (it owns slot k+1) */
  WFM_NOP = 33,        /* placeholder row for the sine slot */
  WFM_COS_ROT = 34     /* cos(w(x-shift)) from the WFM_COS_SINCOS row of equal w;
                          pool: [base_slot, base_shift, D, cos D, sin D] with
                          D ~ w*(base_shift - shift) */
};

/* WfmWave.flags */
#define WFM_WAVE_EXPLICIT_X     0x1u  /* x read from the x array at x_off     */
#define WFM_WAVE_LAST_OVERRIDE  0x2u  /* x[n-1] = x_last (np.linspace endpoint) */
#define WFM_WAVE_CLIP           0x4u  /* np.clip(v, clip_lo, clip_hi) on non-zero segments */
#define WFM_WAVE_PRESHIFT       0x8u  /* x' = x - pre_shift (WaveVStack.shift) */
#define WFM_WAVE_COMPLEX        0x10u /* channel has complex amplitudes        */
#define WFM_WAVE_PAIR           0x20u /* TWO output rows (the I and Q of one mixing() call,
                                         waveform.py:1487-1527) that share their segment table and
                                         every basis-function evaluation: terms flagged
                                         WFM_TERM_PLANE1 sum into the second row (out_off2, offset2).
                                         A pair is real-valued and unclipped. */

/* one output channel (a Waveform, or a whole WaveVStack), or an I/Q pair of them — 112 bytes */
typedef struct WfmWave {
  double   t0;        /* affine grid: x[j] = t0 + j*delta (multiply, then add; never fused) */
  double   delta;
  double   x_last;
  double   clip_lo, clip_hi;
  double   pre_shift;
  double   offset;    /* accumulator start (WaveVStack.offset), 0 otherwise */
  int64_t  n;         /* number of samples */
  int64_t  out_off;   /* index of this channel's first sample in the output buffer */
  int64_t  x_off;     /* index of its first abscissa in the explicit-x buffer */
  int32_t  seg_begin; /* first row in the segment table */
  int32_t  n_seg;     /* rows; the last one has bound +inf */
  uint32_t flags;
  uint32_t reserved;
  int64_t  out_off2;  /* WFM_WAVE_PAIR: first sample of the second row in the output buffer */
  double   offset2;   /* WFM_WAVE_PAIR: accumulator start of the second row */
} WfmWave;

/* per segment: where its distinct factors and its terms start; row n_segs
 * closes the table — 8 bytes */
typedef struct WfmSegPtr {
  int32_t fac;
  int32_t term;
} WfmSegPtr;

/* one distinct basis-function evaluation f(x - shift, args) — 32 bytes */
typedef struct WfmFactor {
  int32_t func;     /* WFM_* id */
  int32_t arg_off;  /* first extra argument in the f64 argument pool */
  double  shift;
  double  a0, a1;   /* the first two scalar arguments, inline */
} WfmFactor;

/* WfmTerm.flags */
#define WFM_TERM_GROUP_END 0x1u /* last term of a stack member: fold the group sum into the channel accumulator */
#define WFM_TERM_PLANE1    0x2u /* the term belongs to the SECOND row of a WFM_WAVE_PAIR channel; within a segment
                                   all first-row terms come before the second-row terms */

/* amp * prod(refs) — 32 bytes */
typedef struct WfmTerm {
  double   amp_re, amp_im;
  int32_t  ref_begin;
  int32_t  n_ref;
  uint32_t flags;
  uint32_t reserved;
} WfmTerm;

/* WfmRef.kind */
#define WFM_POW_ONE  0   /* exponent == 1: multiply by the factor value        */
#define WFM_POW_INT  1   /* small integer exponent: repeated multiplication    */
#define WFM_POW_GEN  2   /* pow(value, expo)                                   */

/* factor-slot ^ exponent — 16 bytes */
typedef struct WfmRef {
  double  expo;
  int32_t slot;   /* index into the segment's factor list */
  int32_t kind;
} WfmRef;

/* WfmProgramDesc.flags */
#define WFM_DESC_DEVICE_TABLES 0x1u /* facs / terms / refs / args are DEVICE pointers (written by wfm_expand_templates):
                                       copied device -> device, their rows are not re-validated on the host; max_rows
                                       must then give the largest number of value rows (factor rows that are not
                                       WFM_NOP) of any segment */

/* host-side view of a lowered batch; all pointers are HOST pointers (but see WFM_DESC_DEVICE_TABLES) */
typedef struct WfmProgramDesc {
  int64_t n_waves;   const WfmWave*   waves;
  int64_t n_segs;    const double*    seg_bound; /* [n_segs] upper bounds        */
                     const WfmSegPtr* seg_ptr;   /* [n_segs + 1]                 */
  int64_t n_facs;    const WfmFactor* facs;
  int64_t n_terms;   const WfmTerm*   terms;
  int64_t n_refs;    const WfmRef*    refs;
  int64_t n_args;    const double*    args;      /* f64 argument / table pool    */
  int64_t n_x;       const double*    x;         /* explicit abscissae (may be NULL) */
  uint32_t flags;    int32_t max_rows;           /* both 0 for plain host tables */
} WfmProgramDesc;

/* ---- pulse templates expanded on the device (see csrc/wfm_expand.cu) ------------------------------------------
 * All pointers of WfmExpandDesc are DEVICE pointers. */
enum { WFM_PATCH_SHIFT = 0, WFM_PATCH_A0 = 1, WFM_PATCH_A1 = 2, WFM_PATCH_ARG = 3, WFM_PATCH_AMP = 4, WFM_PATCH_VALUE = 5 };
typedef struct WfmTemplateDesc {   /* ranges of ONE template in the concatenated template tables — 48 bytes */
  int32_t fac0, n_fac, term0, n_term, ref0, n_ref, arg0, n_arg, patch0, n_patch, rot0, n_rot;
} WfmTemplateDesc;
typedef struct WfmPatch {          /* payload slot j of a pulse goes to entry `index` of table `kind` (template-local) */
  int32_t kind, index;
} WfmPatch;
typedef struct WfmRotRow {         /* a WFM_COS_ROT row of the template: pool block at arg_off (template-local) */
  int32_t fac_row, arg_off;
  double  w, s_b;                  /* constants ... */
  int32_t w_slot, sb_slot;         /* ... unless >= 0: payload slots holding the per-pulse values */
} WfmRotRow;
typedef struct WfmExpandDesc {
  int64_t n_templates;  const WfmTemplateDesc* templates;
  const WfmFactor* t_facs;  const WfmTerm* t_terms;  const WfmRef* t_refs;  const double* t_args;
  const uint8_t* t_has_args;       /* per template factor row: owns a block of the argument pool */
  const WfmPatch* patches;  const WfmRotRow* rots;
  int64_t n_pulses;
  const int32_t* pulse_tmpl;       /* [n_pulses] template of every pulse                         */
  const int32_t* pulse_fac;        /* [n_pulses] first row of the pulse in the expanded tables   */
  const int32_t* pulse_term;  const int32_t* pulse_ref;  const int32_t* pulse_arg;
  int32_t payload_stride;  int32_t reserved;
  const double* payload;           /* [n_pulses][payload_stride]: one double per patch of the pulse's template */
} WfmExpandDesc;
/* writes the rows of every pulse into the DEVICE tables facs / terms / refs / args (sized by the caller) */
int  wfm_expand_templates(const WfmExpandDesc* d, WfmFactor* facs, WfmTerm* terms, WfmRef* refs, double* args,
                          void* stream);

typedef struct WfmProgram* wfm_program_t;

/* output element types */
#define WFM_F64 0
#define WFM_F32 1
#define WFM_F32_FAST 3 /* float output by an fp32 EVALUATOR (fp64 arguments and range reductions, fp32 polynomials,
                          products and sums): ~10 % faster than WFM_F32, which evaluates in fp64 and rounds at the store.
                          Its error is ~1e-7 x (sum of the term magnitudes of a segment): inside 1e-6 of the channel's
                          peak unless large terms cancel (e.g. a DRAG scaling with w * s >> 1).  Opt-in. */
#define WFM_C128 2  /* interleaved (re, im) doubles; assembled from two real planes in scratch that
                       belongs to the program: WFM_C128 launches of ONE program must be stream-ordered */
#define WFM_I16 4   /* 16-bit DAC codes, through wfm_sample_quant / wfm_sample_quant_host only (see there) */

typedef struct WfmLaunch {
  int64_t first_wave;  /* channels [first_wave, first_wave + n_wave) */
  int64_t n_wave;      /* 0 = all from first_wave                    */
  int32_t dtype;       /* WFM_F64 | WFM_F32 | WFM_F32_FAST | WFM_C128 | WFM_I16 */
  int32_t accumulate;  /* 0: out = value; 1: out += value (see below) */
  void*   out;         /* DEVICE pointer (wfm_sample) / HOST pointer (wfm_sample_host) */
  int64_t out_elems;   /* capacity of out, in elements of dtype      */
} WfmLaunch;
/* accumulate = 1 writes out = (OutT)((double)out + v) with ONE rounding, where v is, bit for bit, the value the WFM_F64
 * launch of the same program writes; WFM_F32_FAST then evaluates in fp64 like WFM_F32.  WFM_C128 adds the real and
 * the imaginary part separately.  Flat runs of value 0.0 in programs laid out for the dense kernel may be skipped
 * (out + 0.0 == out), so an out of -0.0 can stay -0.0 there.  Only the samples of the launched channels are read and
 * written.  Host buffers (wfm_sample_host) refuse accumulate (WFM_EUNSUPPORTED); WFM_I16 codes are never accumulated. */

int  wfm_abi_version(void);
const char* wfm_last_error(void);
int  wfm_device_count(void);
int  wfm_trim(void);

/* Uploads the flat IR and runs the device pre-pass.  The host tables may live in
 * pageable or in pinned memory (cudaHostAlloc / torch pin_memory): pinned tables copy
 * at link speed.  Device memory comes from a per-device cache inside the library that
 * wfm_program_destroy returns it to (no cudaMalloc / cudaFree in a scheduler's steady
 * state); wfm_trim() hands the cached blocks back to the driver. */
int  wfm_program_create(const WfmProgramDesc* host_ir, int device, wfm_program_t* out);

/* ---- windowed programs: only some samples of each channel -------------------------------------------------------
 * A window is the samples [j_begin, j_end) of channel `wave`; its sample j goes to out[out_off + (j - j_begin)] (and,
 * for a WFM_WAVE_PAIR channel, the second row's to out[out_off2 + (j - j_begin)]).  The program is laid out as the
 * unwindowed program of the same tables (the same samples per lane, the same tile size, its tiles clipped to the
 * windows) and only the window samples are computed and stored, with the same abscissae and segment ownership.  The
 * values are bit for bit those of the unwindowed program when it evaluates one sample per lane (sparse programs), and
 * otherwise for every window that starts in a segment without factors, at the first sample of a segment or at a tile
 * boundary (the windows of lowering.nonzero_windows): two- and four-sample units rotate a unit's later samples from its first, and a window starting
 * inside a segment starts its units there (the last bits may then differ).  The channel rows' own out_off / out_off2
 * are not used.  Windows must be sorted by (wave, j_begin), must not overlap within a channel, must satisfy
 * 0 <= j_begin < j_end <= n, and their output ranges (both rows of a pair) must be disjoint; j_begin, out_off and
 * out_off2 are multiples of 4 samples (8 for WFM_I16 launches: a window's tiles start at j_begin and at multiples of
 * the tile size, and their stores are 16-byte aligned).  Checked on the host before any device work (WFM_EINVAL).  Complex channels are refused at create, WFM_C128 output and accumulate at launch
 * (WFM_EUNSUPPORTED).  wfm_program_total_samples returns the extent of the windows; first_wave / n_wave of a launch
 * select the windows of those channels.  (The non-zero runs of a batch: lowering.nonzero_windows.) */
typedef struct WfmWindow {  /* 40 bytes */
  int64_t wave, j_begin, j_end;
  int64_t out_off;   /* first output sample of the window */
  int64_t out_off2;  /* WFM_WAVE_PAIR channels: first output sample of the window's second row */
} WfmWindow;
int  wfm_program_create_windows(const WfmProgramDesc* host_ir, const WfmWindow* windows, int64_t n_windows, int device,
                                wfm_program_t* out);
int  wfm_program_destroy(wfm_program_t prog);
int64_t wfm_program_total_samples(wfm_program_t prog);
/* number of kernel launches issued through this program so far */
int64_t wfm_program_launch_count(wfm_program_t prog);
/* how the program was laid out for the sampling kernel: out[0..n) of
 * {tile_samples, packet_buffer_bytes, value_slots, n_tiles, packet_area_bytes,
 *  table_arena_bytes, samples_per_lane_unit, shared_bytes_per_cta}, n <= 8 */
int  wfm_program_info(wfm_program_t prog, int64_t* out, int32_t n);

/* Asynchronous on `stream`.  Large launches of fp64 sparse programs and of every dense
 * program (mostly active samples) deal their tiles dynamically from a per-launch device
 * counter (zeroed on `stream`, guarded by an event of the library): results do not depend
 * on the deal.  Environment WFM_K1_DEAL=static|dynamic overrides for every launch; use
 * `static` when capturing the call into a CUDA graph. */
int  wfm_sample(wfm_program_t prog, const WfmLaunch* launch, void* stream);
int  wfm_sample_host(wfm_program_t prog, const WfmLaunch* launch);

/* ---- 16-bit DAC codes (WFM_I16) ---------------------------------------------------------------------------------
 * Every sample v of an output row with gain g and offset o becomes
 *   code = clamp(rint(v * g + o), -32768, 32767)    multiply, then add (never fused); rint rounds half to even
 *   NaN -> 0;  +inf -> 32767;  -inf -> -32768
 * where v is, bit for bit, the value the WFM_F64 launch of the same program writes (fp64 evaluator, the channel's
 * min / max clip applied first).  Flat segments are converted too: an offset reaches the zero runs.  The conversion
 * runs in the store of the sampling kernel: 2 bytes per sample leave the GPU instead of 8.
 * row_gain_offset is a DEVICE pointer to [n_waves][2 rows][2] doubles (gain, offset), indexed by the program's
 * absolute channel index (first_wave / n_wave sub-launches read their own rows); row 1 is read for WFM_WAVE_PAIR
 * channels only (the second row of the pair).  launch->dtype must be WFM_I16, accumulate 0; complex channels are
 * rejected (WFM_EINVAL), and so is a program whose rows (out_off, out_off2) are not multiples of 8 samples (the
 * 16-byte bulk stores of 2-byte samples; lower such batches with align=8). */
typedef struct WfmQuant {
  const double* row_gain_offset;
} WfmQuant;
int  wfm_sample_quant(wfm_program_t prog, const WfmLaunch* launch, const WfmQuant* quant, void* stream);
int  wfm_sample_quant_host(wfm_program_t prog, const WfmLaunch* launch, const WfmQuant* quant);
/* The same conversion on f64 rows: y[s][j] = code(x[s][j]) with gain_offset[s] = (gain, offset), a DEVICE
 * [n_sig][2] table; x (f64) and y (int16) are DEVICE pointers with their own row strides (in elements). */
int  wfm_quantize(const double* x, int16_t* y, int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                  const double* gain_offset, void* stream);

/* Cascaded biquads, direct form II transposed, exactly scipy.signal.sosfilt:
 *   y = b0*x + z0;  z0 = b1*x - a1*y + z1;  z1 = b2*x - a2*y
 * on `n_sig` independent signals of `n` samples each, signal s starting at
 * x + s*stride (DEVICE pointers, f64; y may alias x).  `sos` is HOST
 * [n_sections][6] (b0 b1 b2 a0 a1 a2), n_sections <= 8.  `initial` is subtracted
 * before and added after filtering (waveform.py:199-203).  `zi` / `zf` are HOST
 * [n_sig][n_sections][2] initial / final states (either may be NULL: zero
 * initial state / final state not returned; a non-NULL zf makes the call
 * synchronous).
 *   WFM_IIR_EXACT  one warp per signal, sequential in time: bit-identical to
 *                  scipy (parallelism = n_sig).
 *   WFM_IIR_SCAN   block-parallel associative scan over time (one CTA per
 *                  signal, 4096-sample tiles): the throughput path; equals the
 *                  sequential result up to the filter's own rounding-noise gain
 *                  (see DESIGN.md, K2). */
#define WFM_IIR_EXACT 0
#define WFM_IIR_SCAN  1
int  wfm_sosfilt(const double* sos, int32_t n_sections, double initial,
                 const double* x, double* y, int64_t n_sig, int64_t n,
                 int64_t stride, const double* zi, double* zf, int32_t mode,
                 void* stream);

/* scipy.signal.lfilter(b, a, x, zi=zi) — one direct-form-II-transposed section of
 * order max(nb, na) - 1 <= 16 (distortion.py:321, the polynomial products built by
 * combine_filters).  One warp per signal, sequential in time, bit-identical to
 * scipy.  b, a, zi, zf are HOST arrays (zi/zf: [n_sig][order], may be NULL; a
 * non-NULL zf makes the call synchronous). */
int  wfm_lfilter(const double* b, int32_t nb, const double* a, int32_t na,
                 const double* x, double* y, int64_t n_sig, int64_t n,
                 int64_t stride, const double* zi, double* zf, void* stream);

/* The same with a mode: WFM_IIR_EXACT = wfm_lfilter; WFM_IIR_SCAN = block-parallel, the scan kernel of wfm_sosfilt
 * (orders 1..4: the DF2T state is a linear system, carries by M x M matrix powers, the samples themselves by scipy's
 * own recurrence from the carried-in state) — equal to the sequential result up to the filter's rounding-noise gain,
 * at the cost of a read and a write (cfg4: 13.4 ms -> 0.3 ms).  Orders above 4 and order 0 run the sequential kernel
 * whatever the mode. */
int  wfm_lfilter_mode(const double* b, int32_t nb, const double* a, int32_t na,
                      const double* x, double* y, int64_t n_sig, int64_t n,
                      int64_t stride, const double* zi, double* zf, int32_t mode, void* stream);

/* y = real(ifft(fft(x) * H)) per signal, H given on the np.fft.fftfreq grid as
 * HOST interleaved complex [n]; arbitrary n.  x, y DEVICE f64 (may alias; signal s
 * of y starts at y + s*stride).  Only the Hermitian part of H contributes to the
 * real part, so signals 2p and 2p+1 share one complex transform (real / imaginary
 * part): a signal's rounding error scales with the larger of its pair, and a
 * non-finite sample in one signal reaches its partner's output too. */
int  wfm_fft_filter(const double* x, double* y, int64_t n_sig, int64_t n,
                    int64_t stride, const double* H, void* stream);

/* A response kept on the device (the kernel convolution of predistort, distortion.py:329-333, applies the same
 * kernel to every batch): wfm_fft_response_create uploads H (HOST interleaved complex [n], np.fft.fftfreq order)
 * once, on the current device; wfm_fft_filter_prepared then computes, for n_sig real signals of n_valid <= n samples
 * each, the first n_valid samples of real(ifft(fft(x zero-padded to n) * H)) — the zero padding of a linear
 * convolution is neither read nor written.  x, y DEVICE f64 with their own pitches (may alias). */
typedef struct WfmFftResponse* wfm_fft_response_t;
int  wfm_fft_response_create(const double* H, int64_t n, wfm_fft_response_t* out);
int  wfm_fft_response_destroy(wfm_fft_response_t r);
int  wfm_fft_filter_prepared(const double* x, double* y, int64_t n_sig, int64_t n_valid,
                             int64_t x_stride, int64_t y_stride, wfm_fft_response_t r, void* stream);

/* reflection (inverse = 0) / correct_reflection (inverse = 1) of distortion.py:208-221:
 * y = real(ifft(fft(x) * H)) resp. / H with H(f) = (1 - A) / (1 - A exp(-2 pi i f tau)) on the
 * np.fft.fftfreq(n, 1 / sample_rate) grid.  The response is built on the device and cached per
 * (device, n, A, tau, sample_rate, inverse): the reference rebuilds it with NumPy on every call.
 * x, y DEVICE f64 with their own pitches (may alias). */
int  wfm_reflection_filter(const double* x, double* y, int64_t n_sig, int64_t n,
                           int64_t x_stride, int64_t y_stride, double A, double tau,
                           double sample_rate, int32_t inverse, void* stream);

/* plain complex DFT of n_sig signals (DEVICE interleaved complex128, in
 * place), forward (sign = -1) or inverse with 1/n scaling (sign = +1) —
 * np.fft.fft / np.fft.ifft. */
int  wfm_fft_c2c(double* data, int64_t n_sig, int64_t n, int64_t stride,
                 int32_t sign, void* stream);

/* ---- calibrations (diagnostics: what bench.py quotes its rooflines against; SURVEY.md 8d) ----
 * wfm_calibrate_fp64: out[0] = fp64 FMA lane-operations per second of the current device
 * (8 independent chains per thread, best of `reps` launches on `stream`), out[1] = ms of one launch.
 * wfm_calibrate_copy: pinned cudaMemcpyAsync ceiling of the current device, dir 0 = device->host,
 * 1 = host->device: out[0] = best GB/s of one copy of `bytes`, out[1] = GB/s over `reps` copies. */
int  wfm_calibrate_fp64(double* out, int32_t reps, void* stream);
int  wfm_calibrate_copy(int64_t bytes, int32_t dir, int32_t reps, double* out);

#ifdef __cplusplus
}
#endif
#endif /* WFM_B200_H */
