// wfm_api.cu — extern "C" boundary of libwfmb200.so (see include/wfm_b200.h).
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <vector>
#include "wfm_internal.h"

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <mutex>
#include <string>
#include <thread>

namespace {

thread_local char g_err[512] = "";

// WFM_TIMING=1: stage times of the host-side entry points on stderr
struct StageTimer {
  bool on;
  const char* what;
  std::chrono::steady_clock::time_point t0;
  explicit StageTimer(const char* w) : on(std::getenv("WFM_TIMING") != nullptr), what(w), t0(std::chrono::steady_clock::now()) {}
  void lap(const char* stage) {
    if (!on) return;
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[wfm] %s: %-22s %8.3f ms\n", what, stage, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define WFM_CUDA(call)                                                                       \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return fail(WFM_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

bool known_func(int f) { return (f >= WFM_LINEAR && f <= WFM_DRAG_SINX) || (f >= WFM_COS_SINCOS && f <= WFM_COS_ROT); }

}  // namespace

// ---- per-device cache of device allocations ------------------------------------------------
// wfm_program_create / wfm_sample_host / wfm_program_destroy run once per batch in a
// scheduler's steady state; cudaMalloc / cudaFree cost milliseconds each and cudaFree
// synchronises the device, so freed blocks are kept and reused (best fit, at most 2x the
// request).  wfm_trim() returns them to the driver.
namespace pool {
struct Block {
  void* p;
  size_t bytes;
};
constexpr int kMaxDevices = 64;
std::mutex mu;
std::vector<Block> cache[kMaxDevices];  // oldest first
size_t cached_bytes[kMaxDevices] = {0};

// at most this much idle device memory is kept per device (WFM_POOL_LIMIT_MB, default 16 GiB of 180)
size_t limit_bytes() {
  static const size_t v = [] {
    const char* s = std::getenv("WFM_POOL_LIMIT_MB");
    const long long mb = s ? std::atoll(s) : 16384;
    return (size_t)std::max<long long>(mb, 0) << 20;
  }();
  return v;
}

size_t round_up(size_t bytes) {
  const size_t g = bytes >= (size_t(1) << 20) ? (size_t(1) << 20) : 4096;  // 1 MiB granules for large blocks
  return (std::max<size_t>(bytes, 1) + g - 1) / g * g;
}

void trim_device(int dev) {
  for (const Block& b : cache[dev]) cudaFree(b.p);
  cache[dev].clear();
  cached_bytes[dev] = 0;
}

// the current device must be `dev`
cudaError_t alloc(int dev, size_t bytes, Block* out) {
  bytes = round_up(bytes);
  if (dev >= 0 && dev < kMaxDevices) {
    std::lock_guard<std::mutex> lk(mu);
    auto& c = cache[dev];
    int best = -1;
    for (int i = 0; i < (int)c.size(); ++i)
      if (c[i].bytes >= bytes && c[i].bytes <= 2 * bytes && (best < 0 || c[i].bytes < c[best].bytes)) best = i;
    if (best >= 0) {
      *out = c[best];
      cached_bytes[dev] -= c[best].bytes;
      c.erase(c.begin() + best);
      return cudaSuccess;
    }
  }
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e == cudaErrorMemoryAllocation && dev >= 0 && dev < kMaxDevices) {
    cudaGetLastError();
    {
      std::lock_guard<std::mutex> lk(mu);
      trim_device(dev);
    }
    e = cudaMalloc(&p, bytes);
  }
  if (e != cudaSuccess) return e;
  *out = Block{p, bytes};
  return cudaSuccess;
}

void release(int dev, const Block& b) {
  if (!b.p) return;
  if (dev < 0 || dev >= kMaxDevices) {
    cudaFree(b.p);
    return;
  }
  std::lock_guard<std::mutex> lk(mu);
  cache[dev].push_back(b);
  cached_bytes[dev] += b.bytes;
  // over the limit: give the oldest idle blocks back to the driver (the caller's device is current)
  while (cached_bytes[dev] > limit_bytes() && !cache[dev].empty()) {
    cudaFree(cache[dev].front().p);
    cached_bytes[dev] -= cache[dev].front().bytes;
    cache[dev].erase(cache[dev].begin());
  }
}
}  // namespace pool

// Small results the host needs from the pre-pass (counters, packet totals) are written by a
// one-thread kernel into MAPPED pinned host memory instead of being copied: a cudaMemcpy D2H
// would queue on the device->host copy engine behind another thread's multi-gigabyte readback.
__global__ void export_words_kernel(const uint32_t* __restrict__ src, volatile uint32_t* dst, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
}
static uint32_t* mapped_scratch() {
  static thread_local uint32_t* p = nullptr;
  if (!p && cudaHostAlloc((void**)&p, 256, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) p = nullptr;
  return p;
}
// n 32-bit words from device memory -> dst (host), complete after the stream is synchronised
static cudaError_t read_words(void* dst_host, const void* src_dev, int n, cudaStream_t st) {
  uint32_t* m = mapped_scratch();
  if (!m) return cudaErrorMemoryAllocation;
  export_words_kernel<<<1, 32, 0, st>>>((const uint32_t*)src_dev, m, n);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) memcpy(dst_host, m, sizeof(uint32_t) * n);
  return e;
}

// Small programs (the README example: two channels, 20 000 samples) are bound by LATENCY: every cudaMemcpyAsync, memset
// and host round trip of wfm_program_create costs microseconds.  Their arena is assembled in one pinned staging buffer
// per host thread and goes up in ONE copy; the tile size comes from the host estimate and is verified after the fact.
constexpr size_t kStageBytes = 256 << 10;
constexpr size_t kBlockingWaitBytes = (size_t)64 << 20;  // wfm_sample_host: device->host copies from this size sleep on an event
static unsigned char* stage_buffer() {
  static thread_local unsigned char* p = nullptr;
  if (!p && cudaHostAlloc((void**)&p, kStageBytes, cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();
    p = nullptr;
  }
  return p;
}
static thread_local bool g_no_fast_create = false;  // set while a fast create is being redone the long way

struct WfmProgram {
  int device = 0;
  wfm::DevProgram dev{};
  std::vector<WfmWave> waves;  // host copy (output sizing, channel ranges)
  pool::Block arena{nullptr, 0};    // every table of the program
  pool::Block tile_tables{nullptr, 0};  // tile rows, packet sizes / offsets (sized once the tile size is chosen)
  pool::Block packets{nullptr, 0};  // the tile packets (sized by the device pre-pass)
  int sizing_passes = 0;
  // one event per stream wfm_sample was called on: destroy waits for exactly that work
  std::vector<std::pair<cudaStream_t, cudaEvent_t>> launch_events;
  std::mutex ev_mu;
  pool::Block stage{nullptr, 0};    // device staging buffer of wfm_sample_host
  wfm::TileDesc* d_tiles = nullptr;
  std::vector<int64_t> tile_prefix;  // tiles before channel w
  // windowed programs (wfm_program_create_windows): the windows and, per channel, its first window ([n_waves + 1])
  bool windowed = false;
  std::vector<WfmWindow> windows;
  std::vector<int64_t> win_first;
  int64_t n_tiles = 0;
  int64_t total_samples = 0;  // extent of the output buffer in samples
  int64_t launches = 0;
  bool any_complex = false;
  bool gapless = false;
  bool rows_aligned8 = true;  // every row starts at a multiple of 8 samples: WFM_I16 output (16-byte stores of 2-byte codes)
  // complex128 output: a planar twin (channels [0, n) = real parts, [n, 2n) = imaginary parts,
  // both real-valued programs for the fast kernel) and the scratch the two planes are sampled into
  WfmProgram* planar = nullptr;
  pool::Block cscratch{nullptr, 0};

  ~WfmProgram() {
    DeviceGuard g(device);
    // kernels launched through this program may still read the tables (cudaFree used to wait
    // for them implicitly): wait for the last launch on every stream that was used — not for
    // the whole device, another thread's copies may be in flight
    for (auto& se : launch_events) {
      cudaEventSynchronize(se.second);
      cudaEventDestroy(se.second);
    }
    delete planar;
    pool::release(device, cscratch);
    pool::release(device, arena);
    pool::release(device, tile_tables);
    pool::release(device, packets);
    pool::release(device, stage);
  }
};

// run fn(lo, hi) over [0, n) on up to 8 host threads; returns the first non-zero result
template <typename F>
static int parallel_ranges(int64_t n, F fn) {
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const int nt = (int)std::min<int64_t>(std::min<unsigned>(hw, 8u), std::max<int64_t>(n / 65536, 1));
  if (nt <= 1) return fn((int64_t)0, n);
  std::vector<int> rc(nt, 0);
  std::vector<std::string> msg(nt);
  std::vector<std::thread> th;
  for (int t = 0; t < nt; ++t)
    th.emplace_back([&, t] {
      rc[t] = fn(n * t / nt, n * (t + 1) / nt);
      if (rc[t] != 0) msg[t] = g_err;  // g_err is thread-local: carry the message to the caller's thread
    });
  for (auto& x : th) x.join();
  for (int t = 0; t < nt; ++t)
    if (rc[t] != 0) return fail(rc[t], "%s", msg[t].c_str());
  return 0;
}

static int validate(const WfmProgramDesc* d, int* max_rows_out) {
  if (!d) return fail(WFM_EINVAL, "null program descriptor");
  const bool dev_tables = (d->flags & WFM_DESC_DEVICE_TABLES) != 0;
  if (d->n_waves < 0 || d->n_segs < 0 || d->n_facs < 0 || d->n_terms < 0 || d->n_refs < 0 || d->n_args < 0 || d->n_x < 0)
    return fail(WFM_EINVAL, "negative table size");
  if (d->n_segs > INT32_MAX - 1 || d->n_facs > INT32_MAX || d->n_terms > INT32_MAX || d->n_refs > INT32_MAX ||
      d->n_args > INT32_MAX)
    return fail(WFM_EINVAL, "table too large for 32-bit indices");
  if ((d->n_waves && !d->waves) || (d->n_segs && (!d->seg_bound || !d->seg_ptr)) || (d->n_facs && !d->facs) ||
      (d->n_terms && !d->terms) || (d->n_refs && !d->refs) || (d->n_args && !d->args) || (d->n_x && !d->x))
    return fail(WFM_EINVAL, "null table pointer with non-zero size");
  if (d->n_segs) {
    const WfmSegPtr e = d->seg_ptr[d->n_segs];
    if (e.fac != d->n_facs || e.term != d->n_terms)
      return fail(WFM_EINVAL, "segment pointer table does not close (%d/%lld factors, %d/%lld terms)", e.fac,
                  (long long)d->n_facs, e.term, (long long)d->n_terms);
  }
  // device-resident tables (wfm_expand_templates wrote them from validated templates): only the host-side tables
  // — channels, segment bounds and pointers — are checked here
  int rc = parallel_ranges(dev_tables ? 0 : d->n_facs, [&](int64_t lo, int64_t hi) {
    for (int64_t k = lo; k < hi; ++k) {
      const WfmFactor& f = d->facs[k];
      if (!known_func(f.func)) return fail(WFM_EUNSUPPORTED, "factor %lld: unknown basis id %d", (long long)k, f.func);
      if (f.arg_off < 0 || f.arg_off > d->n_args)
        return fail(WFM_EINVAL, "factor %lld: argument offset out of range", (long long)k);
      // every basis function's block of the argument pool must lie inside the pool (the device reads
      // it unchecked): layouts as in wfm_basis.cuh / wfm_multidrag.cuh
      const int64_t room = d->n_args - f.arg_off;
      const double* pool = d->args ? d->args + f.arg_off : nullptr;
      auto need = [&](int64_t n) { return n <= room; };
      bool ok = true;
      switch (f.func) {
        case WFM_INTERP: {
          ok = need(2);
          if (ok) {
            const double n = pool[0];
            ok = n >= 1 && n < 2147483647.0 && need(2 + (int64_t)n);
          }
          break;
        }
        case WFM_LINEARCHIRP: ok = need(2); break;
        case WFM_EXPONENTIALCHIRP:
        case WFM_HYPERBOLICCHIRP:
        case WFM_D_GAUSSIAN: ok = need(1); break;
        case WFM_DRAG: ok = need(5); break;
        case WFM_MOLLIFIER:
          if ((int)f.a1 != 0) {
            ok = need(2);
            if (ok) {
              const double nc = pool[1];
              ok = nc >= 0 && nc < 2147483647.0 && need(2 + (int64_t)nc);
            }
          }
          break;
        case WFM_DRAG_SIN:
        case WFM_DRAG_SINX: {
          ok = need(8);
          if (!ok) break;
          const double m = pool[5];
          ok = m >= 0 && m < 1024 && need(8 + 2 * ((int64_t)m + 1));
          if (ok && f.func == WFM_DRAG_SINX) {
            const int64_t tb = 8 + 2 * ((int64_t)m + 1);
            ok = need(tb + 4);
            if (ok && pool[tb + 3] > 0) {
              const double rows = pool[tb + 3];
              ok = rows < 1024 && need(tb + 5);
              if (ok) {
                const double L = pool[tb + 4];
                ok = L >= 0 && L < 65536 && need(tb + 5 + 2 * (int64_t)rows + 2 * (int64_t)rows * (int64_t)L);
              }
            }
          }
          break;
        }
        default: break;
      }
      if (!ok) return fail(WFM_EINVAL, "factor %lld (basis id %d): argument block out of range", (long long)k, f.func);
    }
    return 0;
  });
  if (rc != WFM_OK) return rc;
  // segment table, terms and refs, segment by segment (slot indices are segment-relative)
  std::atomic<int> max_rows{0};
  rc = parallel_ranges(d->n_segs, [&](int64_t lo, int64_t hi) {
    int local_max = 0;
    for (int64_t s = lo; s < hi; ++s) {
      const WfmSegPtr a = d->seg_ptr[s], b = d->seg_ptr[s + 1];
      if (a.fac < 0 || a.term < 0 || b.fac < a.fac || b.term < a.term || b.fac > d->n_facs || b.term > d->n_terms)
        return fail(WFM_EINVAL, "segment %lld: pointer table not monotone", (long long)s);
      const int nf = b.fac - a.fac;
      if (dev_tables) continue;
      int n_values = 0;  // value slots the segment needs: every row but the sine placeholders
      for (int k = 0; k < nf; ++k) {
        const WfmFactor& f = d->facs[a.fac + k];
        n_values += f.func != WFM_NOP;
        if (f.func == WFM_COS_SINCOS) {
          if (k + 1 >= nf || d->facs[a.fac + k + 1].func != WFM_NOP)
            return fail(WFM_EINVAL, "segment %lld: COS_SINCOS row %d needs a NOP row after it", (long long)s, k);
        } else if (f.func == WFM_NOP) {
          if (k == 0 || d->facs[a.fac + k - 1].func != WFM_COS_SINCOS)
            return fail(WFM_EINVAL, "segment %lld: stray NOP row %d", (long long)s, k);
        } else if (f.func == WFM_COS_ROT) {
          if (f.arg_off + 5 > d->n_args) return fail(WFM_EINVAL, "segment %lld: COS_ROT row %d: pool out of range", (long long)s, k);
          const double bs = d->args[f.arg_off];
          const int base = (int)bs;
          if (!(bs >= 0) || base >= k || d->facs[a.fac + base].func != WFM_COS_SINCOS || d->facs[a.fac + base].a0 != f.a0)
            return fail(WFM_EINVAL, "segment %lld: COS_ROT row %d: bad base row", (long long)s, k);
        }
      }
      local_max = std::max(local_max, n_values);
      for (int t = a.term; t < b.term; ++t) {
        const WfmTerm& tm = d->terms[t];
        if (tm.n_ref < 0 || tm.ref_begin < 0 || (int64_t)tm.ref_begin + tm.n_ref > d->n_refs)
          return fail(WFM_EINVAL, "term %d: reference range out of bounds", t);
        // the sampling kernel walks a segment's references as ONE contiguous slice: packed in term order
        if (t + 1 < d->n_terms && d->terms[t + 1].ref_begin != tm.ref_begin + tm.n_ref)
          return fail(WFM_EINVAL, "term %d: references must be packed in term order", t + 1);
        for (int r = tm.ref_begin; r < tm.ref_begin + tm.n_ref; ++r) {
          const WfmRef& rf = d->refs[r];
          if (rf.slot < 0 || rf.slot >= nf) return fail(WFM_EINVAL, "ref %d: slot %d outside segment (%d factors)", r, rf.slot, nf);
          if (d->facs[a.fac + rf.slot].func == WFM_NOP) return fail(WFM_EINVAL, "ref %d: refers to a NOP row", r);
          if (rf.kind < WFM_POW_ONE || rf.kind > WFM_POW_GEN) return fail(WFM_EINVAL, "ref %d: bad exponent kind", r);
        }
      }
      if (b.term > a.term && !(d->terms[b.term - 1].flags & WFM_TERM_GROUP_END))
        return fail(WFM_EINVAL, "segment %lld: last term does not close its group", (long long)s);
      // I/Q pairs: the first row's terms, then the second row's; the first row ends on a closed group
      for (int t = a.term + 1; t < b.term; ++t) {
        const bool p_prev = d->terms[t - 1].flags & WFM_TERM_PLANE1, p_cur = d->terms[t].flags & WFM_TERM_PLANE1;
        if (p_prev && !p_cur) return fail(WFM_EINVAL, "segment %lld: second-row terms must follow the first row's", (long long)s);
        if (!p_prev && p_cur && !(d->terms[t - 1].flags & WFM_TERM_GROUP_END))
          return fail(WFM_EINVAL, "segment %lld: the first row's last term does not close its group", (long long)s);
      }
    }
    int cur = max_rows.load();
    while (local_max > cur && !max_rows.compare_exchange_weak(cur, local_max)) {
    }
    return 0;
  });
  if (rc != WFM_OK) return rc;
  *max_rows_out = dev_tables ? d->max_rows : max_rows.load();
  if (dev_tables && (d->max_rows < 0 || d->max_rows > 4096)) return fail(WFM_EINVAL, "max_rows out of range");
  for (int64_t w = 0; w < d->n_waves; ++w) {
    const WfmWave& wv = d->waves[w];
    if (wv.n < 0 || wv.out_off < 0) return fail(WFM_EINVAL, "channel %lld: negative extent", (long long)w);
    if (wv.n >= INT32_MAX) return fail(WFM_EINVAL, "channel %lld: more than 2^31-2 samples", (long long)w);
    if (wv.n_seg < 1 || wv.seg_begin < 0 || (int64_t)wv.seg_begin + wv.n_seg > d->n_segs)
      return fail(WFM_EINVAL, "channel %lld: segment range out of bounds", (long long)w);
    if (!(d->seg_bound[wv.seg_begin + wv.n_seg - 1] == INFINITY))
      return fail(WFM_EINVAL, "channel %lld: last bound must be +inf", (long long)w);
    if ((wv.flags & WFM_WAVE_EXPLICIT_X) && (wv.x_off < 0 || wv.x_off + wv.n > d->n_x))
      return fail(WFM_EINVAL, "channel %lld: explicit abscissae out of range", (long long)w);
    if (wv.out_off % 4) return fail(WFM_EINVAL, "channel %lld: out_off must be a multiple of 4 (16-byte stores)", (long long)w);
    if (dev_tables && (wv.flags & WFM_WAVE_COMPLEX))
      return fail(WFM_EUNSUPPORTED, "channel %lld: complex amplitudes need host tables (the planar twin is built from them)", (long long)w);
    if (wv.flags & WFM_WAVE_PAIR) {
      if (wv.out_off2 < 0 || wv.out_off2 % 4) return fail(WFM_EINVAL, "channel %lld: out_off2 must be a non-negative multiple of 4", (long long)w);
      if (wv.flags & (WFM_WAVE_CLIP | WFM_WAVE_COMPLEX))
        return fail(WFM_EINVAL, "channel %lld: an I/Q pair is real-valued and unclipped", (long long)w);
      const int64_t lo = std::min(wv.out_off, wv.out_off2), hi = std::max(wv.out_off, wv.out_off2);
      if (lo + wv.n > hi) return fail(WFM_EINVAL, "channel %lld: the two rows of the pair overlap", (long long)w);
    }
  }
  return WFM_OK;
}

// the windows of wfm_program_create_windows, checked against the (validated) channel table; win_first[w] = first window
// of channel w, win_first[n_waves] = n_windows
static int validate_windows(const WfmProgramDesc* d, const WfmWindow* win, int64_t n, std::vector<int64_t>* win_first) {
  if (n < 0 || (n > 0 && !win)) return fail(WFM_EINVAL, "bad window table");
  win_first->assign(d->n_waves + 1, n);
  std::vector<std::pair<int64_t, int64_t>> ranges;  // output ranges of every window row
  ranges.reserve(n);
  for (int64_t i = n - 1; i >= 0; --i) {
    const WfmWindow& v = win[i];
    if (v.wave < 0 || v.wave >= d->n_waves) return fail(WFM_EINVAL, "window %lld: channel %lld out of range", (long long)i, (long long)v.wave);
    const WfmWave& w = d->waves[v.wave];
    if (!(0 <= v.j_begin && v.j_begin < v.j_end && v.j_end <= w.n))
      return fail(WFM_EINVAL, "window %lld: [%lld, %lld) is not inside [0, %lld) or is empty", (long long)i, (long long)v.j_begin,
                  (long long)v.j_end, (long long)w.n);
    if (i + 1 < n && (win[i + 1].wave < v.wave || (win[i + 1].wave == v.wave && win[i + 1].j_begin < v.j_end)))
      return fail(WFM_EINVAL, "window %lld: windows must be sorted by (wave, j_begin) and must not overlap", (long long)i + 1);
    (*win_first)[v.wave] = i;
    if (v.out_off < 0 || v.out_off % 4) return fail(WFM_EINVAL, "window %lld: out_off must be a non-negative multiple of 4", (long long)i);
    // a window's tiles start at j_begin and at multiples of the tile size: their outputs stay 16-byte aligned
    if (v.j_begin % 4) return fail(WFM_EINVAL, "window %lld: j_begin must be a multiple of 4", (long long)i);
    ranges.emplace_back(v.out_off, v.out_off + (v.j_end - v.j_begin));
    if (w.flags & WFM_WAVE_PAIR) {
      if (v.out_off2 < 0 || v.out_off2 % 4) return fail(WFM_EINVAL, "window %lld: out_off2 must be a non-negative multiple of 4", (long long)i);
      ranges.emplace_back(v.out_off2, v.out_off2 + (v.j_end - v.j_begin));
    }
  }
  for (int64_t w = d->n_waves - 1; w >= 0; --w) (*win_first)[w] = std::min((*win_first)[w], (*win_first)[w + 1]);
  std::sort(ranges.begin(), ranges.end());
  for (size_t k = 1; k < ranges.size(); ++k)
    if (ranges[k].first < ranges[k - 1].second)
      return fail(WFM_EINVAL, "window output ranges intersect at sample %lld", (long long)ranges[k].first);
  return WFM_OK;
}

// [lo, hi): the output samples the channels [first, first + count) write (lo = INT64_MAX, hi = 0 if none)
static void output_extent(const WfmProgram* prog, int64_t first, int64_t count, int64_t* lo, int64_t* hi) {
  *lo = INT64_MAX;
  *hi = 0;
  if (!prog->windowed) {
    for (int64_t w = first; w < first + count; ++w) {
      *lo = std::min(*lo, prog->waves[w].out_off);
      *hi = std::max(*hi, prog->waves[w].out_off + prog->waves[w].n);
      if (prog->waves[w].flags & WFM_WAVE_PAIR) *hi = std::max(*hi, prog->waves[w].out_off2 + prog->waves[w].n);
    }
    return;
  }
  for (int64_t i = prog->win_first[first]; i < prog->win_first[first + count]; ++i) {
    const WfmWindow& v = prog->windows[i];
    const int64_t len = v.j_end - v.j_begin;
    *lo = std::min(*lo, v.out_off);
    *hi = std::max(*hi, v.out_off + len);
    if (prog->waves[v.wave].flags & WFM_WAVE_PAIR) {
      *lo = std::min(*lo, v.out_off2);
      *hi = std::max(*hi, v.out_off2 + len);
    }
  }
}

static int create_program(const WfmProgramDesc* d, const WfmWindow* windows, int64_t n_windows, int device, wfm_program_t* out);

extern "C" {

int wfm_abi_version(void) { return WFM_ABI_VERSION; }

const char* wfm_last_error(void) { return g_err; }

int wfm_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int wfm_trim(void) {
  std::lock_guard<std::mutex> lk(pool::mu);
  int prev = -1;
  cudaGetDevice(&prev);
  for (int dev = 0; dev < pool::kMaxDevices; ++dev) {
    if (pool::cache[dev].empty()) continue;
    if (cudaSetDevice(dev) == cudaSuccess) pool::trim_device(dev);
  }
  if (prev >= 0) cudaSetDevice(prev);
  cudaGetLastError();
  return WFM_OK;
}

int wfm_program_create(const WfmProgramDesc* d, int device, wfm_program_t* out) {
  return create_program(d, nullptr, -1, device, out);
}

int wfm_program_create_windows(const WfmProgramDesc* d, const WfmWindow* windows, int64_t n_windows, int device,
                               wfm_program_t* out) {
  if (n_windows < 0) return fail(WFM_EINVAL, "negative window count");
  return create_program(d, windows, n_windows, device, out);
}

}  // extern "C"

// n_windows < 0: the plain program (every sample of every channel)
static int create_program(const WfmProgramDesc* d, const WfmWindow* windows, int64_t n_windows, int device, wfm_program_t* out) {
  if (!out) return fail(WFM_EINVAL, "null output handle");
  *out = nullptr;
  StageTimer tm("program_create");
  const bool windowed = n_windows >= 0;
  // all device work of this call runs on the calling thread's own stream: two host threads
  // (a scheduler double-buffering its batches) overlap one batch's upload and pre-pass with
  // the other's device->host copy instead of serialising on the legacy default stream
  const cudaStream_t ST = cudaStreamPerThread;
  int max_rows = 0;
  int rc = validate(d, &max_rows);
  if (rc != WFM_OK) return rc;
  std::vector<int64_t> win_first;
  if (windowed) {
    rc = validate_windows(d, windows, n_windows, &win_first);
    if (rc != WFM_OK) return rc;
    for (int64_t w = 0; w < d->n_waves; ++w)
      if (d->waves[w].flags & WFM_WAVE_COMPLEX)
        return fail(WFM_EUNSUPPORTED, "channel %lld: a windowed program samples real channels only", (long long)w);
  }
  tm.lap("validate");
  DeviceGuard g(device);
  if (!g.ok) return fail(WFM_ECUDA, "cannot select CUDA device %d: %s", device, cudaGetErrorString(cudaGetLastError()));
  WfmProgram* p = new (std::nothrow) WfmProgram();
  if (!p) return fail(WFM_ENOMEM, "out of host memory");
  p->device = device;
  p->waves.assign(d->waves, d->waves + d->n_waves);
  if (windowed) {
    p->windowed = true;
    p->windows.assign(windows, windows + n_windows);
    p->win_first = std::move(win_first);
  }
  p->dev.n_slots = 1 + std::max(1, std::min(max_rows, wfm::kMaxSlots));
  p->dev.planes = 1;
  p->dev.dense = 0;

  int64_t samples = 0, total = 0, rows = 0;
  for (int64_t w = 0; w < d->n_waves; ++w) {
    samples += d->waves[w].n;
    rows += d->waves[w].n * ((d->waves[w].flags & WFM_WAVE_PAIR) ? 2 : 1);
    total = std::max(total, d->waves[w].out_off + d->waves[w].n);
    if (d->waves[w].flags & WFM_WAVE_COMPLEX) p->any_complex = true;
    if (d->waves[w].out_off % 8) p->rows_aligned8 = false;
    if (d->waves[w].flags & WFM_WAVE_PAIR) {
      p->dev.planes = 2;
      total = std::max(total, d->waves[w].out_off2 + d->waves[w].n);
      if (d->waves[w].out_off2 % 8) p->rows_aligned8 = false;
    }
  }
  // A windowed program is laid out as the plain program of the same channels: the same unit and tile size (decided
  // from the channels' samples), its tiles the plain tiles clipped to the windows.  Two- and four-sample units pair
  // the samples of a segment from the start of its tile and rotate the second sample's sines from the first's, so only
  // the plain program's tiles give the plain program's values.  Only the output rows are the windows'.
  if (windowed) {
    rows = 0;
    for (const WfmWindow& v : p->windows)
      rows += (v.j_end - v.j_begin) * ((d->waves[v.wave].flags & WFM_WAVE_PAIR) ? 2 : 1);
    int64_t lo;
    output_extent(p, 0, d->n_waves, &lo, &total);
    p->rows_aligned8 = true;
    for (const WfmWindow& v : p->windows)
      if (v.j_begin % 8 || v.out_off % 8 || ((d->waves[v.wave].flags & WFM_WAVE_PAIR) && v.out_off2 % 8)) p->rows_aligned8 = false;
  }
  p->total_samples = total;
  p->gapless = rows == total;  // the channels' rows tile the output: nothing between them that the kernel leaves unwritten

  // arena 1: every table that does not depend on the tile size (ABI tables + segment plans), 256-byte aligned slots
  size_t arena_bytes = 0;
  auto reserve = [&](size_t bytes) {
    const size_t off = arena_bytes;
    arena_bytes += (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255;
    return off;
  };
  const size_t o_waves = reserve(sizeof(WfmWave) * d->n_waves), o_bound = reserve(sizeof(double) * d->n_segs),
               o_segptr = reserve(sizeof(WfmSegPtr) * (d->n_segs + 1)), o_facs = reserve(sizeof(WfmFactor) * d->n_facs),
               o_terms = reserve(sizeof(WfmTerm) * d->n_terms), o_refs = reserve(sizeof(WfmRef) * d->n_refs),
               o_args = reserve(sizeof(double) * d->n_args), o_x = reserve(sizeof(double) * d->n_x),
               o_segwave = reserve(sizeof(int32_t) * d->n_segs), o_segstart = reserve(sizeof(int32_t) * d->n_segs),
               o_segval = reserve(sizeof(double) * d->n_segs),
               o_segval1 = reserve(p->dev.planes == 2 ? sizeof(double) * d->n_segs : 0), o_plan = reserve(sizeof(wfm::SegPlan) * d->n_segs),
               o_rowslot = reserve((size_t)d->n_facs), o_cterms = reserve(sizeof(wfm::CTerm) * d->n_terms),
               o_prefix = reserve(sizeof(int64_t) * (std::max<int64_t>(d->n_waves, windowed ? n_windows : 0) + 1)), o_stats = reserve(sizeof(uint64_t) * 2),
               o_windows = reserve(windowed ? sizeof(WfmWindow) * n_windows : 0);
  cudaError_t e = pool::alloc(device, arena_bytes, &p->arena);
  if (e != cudaSuccess) {
    delete p;
    return fail(e == cudaErrorMemoryAllocation ? WFM_ENOMEM : WFM_ECUDA, "allocating %zu bytes for the program failed: %s",
                arena_bytes, cudaGetErrorString(e));
  }
  char* base = (char*)p->arena.p;
  const bool small_program = samples <= (int64_t)1 << 20;
  const char* force_unit = std::getenv("WFM_K1_UNIT");
  const bool unit_forced = force_unit && (force_unit[0] == '1' || force_unit[0] == '2' || force_unit[0] == '4');
  // the fast path of small programs: the whole arena staged and sent in one copy, no sizing round trip (a windowed
  // program measures the plain tiles to take their size)
  unsigned char* stg = (small_program && !windowed && !g_no_fast_create && !(d->flags & WFM_DESC_DEVICE_TABLES) && !p->any_complex &&
                        arena_bytes <= kStageBytes && d->n_waves > 0 && !std::getenv("WFM_NO_FAST_CREATE"))
                           ? stage_buffer() : nullptr;
  auto up = [&](size_t off, const void* host, size_t bytes) {
    if (bytes == 0) return;
    if (stg) {
      memcpy(stg + off, host, bytes);
      return;
    }
    // pinned host tables (cudaHostAlloc / torch pin_memory) copy at link speed; pageable ones are staged by the driver
    if (e == cudaSuccess) e = cudaMemcpyAsync(base + off, host, bytes, cudaMemcpyHostToDevice, ST);
  };
  up(o_waves, d->waves, sizeof(WfmWave) * d->n_waves);
  up(o_bound, d->seg_bound, sizeof(double) * d->n_segs);
  up(o_segptr, d->seg_ptr, d->n_segs ? sizeof(WfmSegPtr) * (d->n_segs + 1) : 0);
  if (d->flags & WFM_DESC_DEVICE_TABLES) {
    // written on this device by wfm_expand_templates, on a stream the caller has ordered before this call
    auto dd = [&](size_t off, const void* src, size_t bytes) {
      if (e == cudaSuccess && bytes > 0) e = cudaMemcpyAsync(base + off, src, bytes, cudaMemcpyDeviceToDevice, ST);
    };
    dd(o_facs, d->facs, sizeof(WfmFactor) * d->n_facs);
    dd(o_terms, d->terms, sizeof(WfmTerm) * d->n_terms);
    dd(o_refs, d->refs, sizeof(WfmRef) * d->n_refs);
    dd(o_args, d->args, sizeof(double) * d->n_args);
  } else {
    up(o_facs, d->facs, sizeof(WfmFactor) * d->n_facs);
    up(o_terms, d->terms, sizeof(WfmTerm) * d->n_terms);
    up(o_refs, d->refs, sizeof(WfmRef) * d->n_refs);
    up(o_args, d->args, sizeof(double) * d->n_args);
  }
  up(o_x, d->x, sizeof(double) * d->n_x);
  if (windowed) up(o_windows, windows, sizeof(WfmWindow) * n_windows);
  p->dev.waves = (const WfmWave*)(base + o_waves);
  p->dev.seg_bound = (const double*)(base + o_bound);
  p->dev.seg_ptr = (const WfmSegPtr*)(base + o_segptr);
  p->dev.facs = (const WfmFactor*)(base + o_facs);
  p->dev.terms = (const WfmTerm*)(base + o_terms);
  p->dev.refs = (const WfmRef*)(base + o_refs);
  p->dev.args = (const double*)(base + o_args);
  p->dev.x = (const double*)(base + o_x);
  p->dev.seg_wave = (const int32_t*)(base + o_segwave);
  p->dev.seg_start = (const int32_t*)(base + o_segstart);
  p->dev.seg_val = (const double*)(base + o_segval);
  p->dev.seg_val1 = p->dev.planes == 2 ? (const double*)(base + o_segval1) : nullptr;
  p->dev.seg_plan = (const wfm::SegPlan*)(base + o_plan);
  p->dev.row_slot = (const uint8_t*)(base + o_rowslot);
  p->dev.cterms = (const wfm::CTerm*)(base + o_cterms);
  tm.lap("arena + uploads");

  // device pre-pass 1a: owning channel of every segment, segment start positions and flat
  // values, segment plans
  wfm::PrepareBuffers pb{(int32_t*)(base + o_segwave), (int32_t*)(base + o_segstart), (double*)(base + o_segval),
                         p->dev.planes == 2 ? (double*)(base + o_segval1) : nullptr, (wfm::SegPlan*)(base + o_plan), (uint8_t*)(base + o_rowslot), (wfm::CTerm*)(base + o_cterms),
                         nullptr, windowed ? (const WfmWindow*)(base + o_windows) : nullptr, (const int64_t*)(base + o_prefix),
                         nullptr};
  wfm::PrepareCounts pc{d->n_waves, d->n_segs, d->n_facs, d->n_terms, 0, windowed ? n_windows : 0};
  p->dev.unit = 1;
  uint32_t* d_stats = (uint32_t*)(base + o_stats);
  auto cap_of = [&](int ts) { return wfm::packet_capacity(p->dev, ts); };
  // the largest tile the average packet density allows (the device then measures every tile)
  auto estimate_tile = [&]() {
    int ts = wfm::kMaxTileSamples;
    const double per_sample = samples > 0 ? 1.0 / (double)samples : 0.0;
    const double ir = ((double)d->n_facs * 28.0 /* SRow, CRow, GRow: 32 bytes each; NOP rows vanish */ +
                       (double)d->n_terms * sizeof(wfm::CTerm) + (double)d->n_segs * sizeof(wfm::ARow)) * per_sample;
    while (ts > wfm::kMinTileSamples && !(cap_of(ts) >= 256 && 64.0 + ir * ts <= cap_of(ts))) ts -= 128;
    return ts;
  };
  // n_plain / plain_prefix: the plain program's tiles (what the tile size is measured on); n_tiles / p->tile_prefix: this
  // program's (a windowed program's: per window the grid cells it intersects, range_prefix; per channel, tile_prefix)
  int64_t n_tiles = 0, n_plain = 0;
  std::vector<int64_t> plain_prefix, range_prefix;
  auto set_tile = [&](int ts) {
    p->dev.tile_samples = ts;
    p->dev.pkt_cap = std::max(cap_of(ts), 64);
    plain_prefix.resize(d->n_waves + 1);
    n_plain = 0;
    for (int64_t w = 0; w < d->n_waves; ++w) {
      plain_prefix[w] = n_plain;
      n_plain += (d->waves[w].n + ts - 1) / ts;
    }
    plain_prefix[d->n_waves] = n_plain;
    if (!windowed) {
      p->tile_prefix = plain_prefix;
      n_tiles = n_plain;
      return;
    }
    range_prefix.resize(n_windows + 1);
    n_tiles = 0;
    for (int64_t i = 0; i < n_windows; ++i) {
      range_prefix[i] = n_tiles;
      n_tiles += (p->windows[i].j_end - 1) / ts - p->windows[i].j_begin / ts + 1;
    }
    range_prefix[n_windows] = n_tiles;
    p->tile_prefix.resize(d->n_waves + 1);
    for (int64_t w = 0; w <= d->n_waves; ++w) p->tile_prefix[w] = range_prefix[p->win_first[w]];
  };
  // the device's tile_prefix: this program's tiles, or (plain = true) the plain program's
  auto upload_prefix = [&](bool plain) {
    if (windowed && !plain) up(o_prefix, range_prefix.data(), sizeof(int64_t) * (n_windows + 1));
    else up(o_prefix, plain_prefix.data(), sizeof(int64_t) * (d->n_waves + 1));
  };
  if (stg) {
    // everything the device needs is known on the host: unit, tile size, tile prefix; zeroed statistics ride along
    if (unit_forced) p->dev.unit = force_unit[0] - '0';
    p->dev.dense = p->dev.unit == wfm::kDenseUnit ? 1 : 0;
    set_tile(estimate_tile());
    upload_prefix(false);
    memset(stg + o_stats, 0, sizeof(uint64_t) * 2);
    e = cudaMemcpyAsync(base, stg, arena_bytes, cudaMemcpyHostToDevice, ST);
  }
  if (e == cudaSuccess) e = wfm::launch_prepare_segments(p->dev, pc, pb, ST);

  // Unit: samples per lane and evaluation.  Dense programs (more than two rounds of 32 active
  // samples in an average 1024-sample tile) evaluate two samples per lane, sparse ones one.
  // (Small programs skip the question and its round trip to the host: their figure of merit is latency — the README
  // example is 20 000 samples — and the unit size only tunes throughput.)
  if (!stg) {
    if (unit_forced) {
      p->dev.unit = force_unit[0] - '0';
    } else if (small_program) {
      p->dev.unit = 1;
    } else {
      unsigned long long active = 0;
      unsigned long long* d_active = (unsigned long long*)(base + o_stats);
      if (e == cudaSuccess) e = cudaMemsetAsync(d_active, 0, sizeof(active), ST);
      if (e == cudaSuccess) e = wfm::launch_count_active(p->dev, d->n_segs, d_active, ST);
      if (e == cudaSuccess) e = read_words(&active, d_active, 2, ST);
      if (samples > 0 && (double)active * 2.0 > (double)samples) p->dev.unit = wfm::kDenseUnit;  // mostly active: dense kernel
      else p->dev.unit = (samples > 0 && (double)active * 1024.0 > 64.0 * (double)samples) ? 2 : 1;
    }
    p->dev.dense = p->dev.unit == wfm::kDenseUnit ? 1 : 0;
  }

  // Tile size.  A warp's slice of shared memory holds the output tile (8 B per sample), the
  // value slots and two packet buffers.  Take the LARGEST tile (a multiple of 128 samples)
  // for which every tile's packet fits its buffer, measured on the device: start from the
  // size the average packet density allows and step down while more than 1 tile in 4096 would
  // not fit (those take the kernel's cold path).
  int ts = stg ? p->dev.tile_samples : estimate_tile();
  int sizing_passes = 0;
  for (; !stg; ts -= 128) {
    set_tile(ts);
    if (std::max(n_tiles, n_plain) >= INT32_MAX) {
      delete p;
      return fail(WFM_EINVAL, "too many tiles (%lld)", (long long)std::max(n_tiles, n_plain));
    }
    if (e != cudaSuccess || ts <= wfm::kMinTileSamples || n_plain == 0) break;
    // sizing pass on the plain tiles: statistics only
    uint32_t stats[2] = {0, 0};
    e = cudaMemsetAsync(d_stats, 0, sizeof(stats), ST);
    upload_prefix(true);
    wfm::PrepareBuffers pb_plain = pb;
    pb_plain.windows = nullptr;
    wfm::PrepareCounts pc_plain = pc;
    pc_plain.n_tiles = n_plain;
    if (e == cudaSuccess) e = wfm::launch_prepare_tiles(p->dev, pc_plain, pb_plain, d_stats, ST);
    if (e == cudaSuccess) e = read_words(stats, d_stats, 2, ST);  // synchronises: tile_prefix may be rewritten now
    ++sizing_passes;
    if (e != cudaSuccess || (int64_t)stats[1] * 4096 <= n_plain) break;
  }
  p->n_tiles = n_tiles;
  p->sizing_passes = sizing_passes;
  tm.lap("device pre-pass 1 (tile size)");

  // arena 2: the tile tables
  size_t tiles_bytes = 0;
  auto reserve2 = [&](size_t bytes) {
    const size_t off = tiles_bytes;
    tiles_bytes += (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255;
    return off;
  };
  const size_t nt1 = (size_t)n_tiles + 1;
  const size_t o_tiles = reserve2(sizeof(wfm::TileDesc) * n_tiles), o_pktsize = reserve2(sizeof(uint32_t) * nt1),
               o_pktoff = reserve2(sizeof(uint32_t) * nt1), o_scratch = reserve2(sizeof(uint32_t) * (nt1 / 4096 + 2));
  if (e == cudaSuccess) e = pool::alloc(device, tiles_bytes, &p->tile_tables);
  char* base2 = (char*)p->tile_tables.p;
  uint32_t total16 = 0;
  if (e == cudaSuccess) {
    p->d_tiles = (wfm::TileDesc*)(base2 + o_tiles);
    p->dev.pkt_off = (const uint32_t*)(base2 + o_pktoff);
    pb.tiles = p->d_tiles;
    pb.pkt_size = (uint32_t*)(base2 + o_pktsize);
    pc.n_tiles = n_tiles;
    if (!stg) upload_prefix(false);
    // pre-pass 1b: the tile rows with their packet sizes (fast path: and the statistics the sizing pass would have
    // taken); then the packet offsets
    if (e == cudaSuccess) e = wfm::launch_prepare_tiles(p->dev, pc, pb, stg ? d_stats : nullptr, ST);
    if (e == cudaSuccess)
      e = wfm::launch_scan((uint32_t*)(base2 + o_pktsize), (uint32_t*)(base2 + o_pktoff), (uint32_t*)(base2 + o_scratch),
                           n_tiles, ST);
    // the packet area: its exact size comes from the scan; a small program takes the upper bound (no packet exceeds its
    // buffer: larger tiles are cold, header only) and saves the round trip
    if (small_program && (size_t)n_tiles * (size_t)std::max(p->dev.pkt_cap, 96) <= ((size_t)4 << 20))
      total16 = (uint32_t)(((size_t)n_tiles * (size_t)std::max(p->dev.pkt_cap, 96) + 15) / 16);
    else if (e == cudaSuccess) e = read_words(&total16, (uint32_t*)(base2 + o_pktoff) + n_tiles, 1, ST);
  }
  tm.lap("device pre-pass 1 (tiles)");
  // pass 2: the packets themselves
  if (e == cudaSuccess) e = pool::alloc(device, std::max<size_t>((size_t)total16 * 16, 16), &p->packets);
  p->dev.packets = (const unsigned char*)p->packets.p;
  if (e == cudaSuccess) e = wfm::launch_fill_packets(p->dev, p->d_tiles, n_tiles, pc, pb, (unsigned char*)p->packets.p, ST);
  if (stg && n_tiles > 0 && ts > wfm::kMinTileSamples) {
    // the one synchronisation of the fast path also brings the statistics: tiles whose packet does not fit their buffer
    // (they would take the kernel's cold path) send the program through the measured sizing loop instead
    uint32_t stats[2] = {0, 0};
    if (e == cudaSuccess) e = read_words(stats, d_stats, 2, ST);
    if (e == cudaSuccess && (int64_t)stats[1] * 4096 > n_tiles) {
      delete p;
      g_no_fast_create = true;
      const int rc2 = create_program(d, windows, n_windows, device, out);
      g_no_fast_create = false;
      return rc2;
    }
  } else if (e == cudaSuccess) {
    e = cudaStreamSynchronize(ST);
  }
  tm.lap("device pre-pass 2");
  if (e != cudaSuccess) {
    delete p;
    return fail(WFM_ECUDA, "uploading the program failed: %s", cudaGetErrorString(e));
  }
  if (p->any_complex) {
    // the planar twin: every table twice, the second copy's amplitudes = the imaginary parts
    const int64_t nw = d->n_waves, ns = d->n_segs, nf = d->n_facs, nt = d->n_terms, nr = d->n_refs;
    std::vector<WfmWave> waves2(2 * nw);
    std::vector<double> bound2(2 * ns);
    std::vector<WfmSegPtr> segptr2(2 * ns + 1);
    std::vector<WfmFactor> facs2(2 * nf);
    std::vector<WfmTerm> terms2(2 * nt);
    std::vector<WfmRef> refs2(2 * nr);
    for (int c = 0; c < 2; ++c) {
      for (int64_t w = 0; w < nw; ++w) {
        WfmWave v = d->waves[w];
        v.flags &= ~(uint32_t)WFM_WAVE_COMPLEX;
        v.seg_begin += (int32_t)(c * ns);
        v.out_off += c * ((total + 3) & ~(int64_t)3);  // planes stay 16-byte aligned
        v.out_off2 += c * ((total + 3) & ~(int64_t)3);
        if (c == 1) {
          v.offset = 0.0;  // offsets and clipping act on the real part
          v.flags &= ~(uint32_t)WFM_WAVE_CLIP;
        }
        waves2[c * nw + w] = v;
      }
      for (int64_t k = 0; k < ns; ++k) {
        bound2[c * ns + k] = d->seg_bound[k];
        segptr2[c * ns + k] = WfmSegPtr{(int32_t)(d->seg_ptr[k].fac + c * nf), (int32_t)(d->seg_ptr[k].term + c * nt)};
      }
      for (int64_t k = 0; k < nf; ++k) facs2[c * nf + k] = d->facs[k];  // argument pool and abscissae are shared
      for (int64_t k = 0; k < nt; ++k) {
        WfmTerm t = d->terms[k];
        if (c == 1) t.amp_re = t.amp_im;
        t.amp_im = 0.0;
        t.ref_begin += (int32_t)(c * nr);
        terms2[c * nt + k] = t;
      }
      for (int64_t k = 0; k < nr; ++k) refs2[c * nr + k] = d->refs[k];
    }
    segptr2[2 * ns] = WfmSegPtr{(int32_t)(2 * nf), (int32_t)(2 * nt)};
    WfmProgramDesc d2 = *d;
    d2.n_waves = 2 * nw; d2.waves = waves2.data();
    d2.n_segs = 2 * ns; d2.seg_bound = bound2.data(); d2.seg_ptr = segptr2.data();
    d2.n_facs = 2 * nf; d2.facs = facs2.data();
    d2.n_terms = 2 * nt; d2.terms = terms2.data();
    d2.n_refs = 2 * nr; d2.refs = refs2.data();
    if (2 * (double)ns > INT32_MAX - 2 || 2 * (double)nf > INT32_MAX || 2 * (double)nt > INT32_MAX || 2 * (double)nr > INT32_MAX) {
      delete p;
      return fail(WFM_EINVAL, "complex program too large for 32-bit indices once split into planes");
    }
    const int rc2 = wfm_program_create(&d2, device, &p->planar);
    if (rc2 != WFM_OK) {
      delete p;
      return rc2;
    }
    tm.lap("planar twin (complex output)");
  }
  *out = p;
  return WFM_OK;
}

extern "C" {

int wfm_program_destroy(wfm_program_t prog) {
  StageTimer tm("program_destroy");
  delete prog;
  tm.lap("release");
  return WFM_OK;
}

int64_t wfm_program_total_samples(wfm_program_t prog) { return prog ? prog->total_samples : -1; }

int64_t wfm_program_launch_count(wfm_program_t prog) { return prog ? prog->launches : -1; }

int wfm_program_info(wfm_program_t prog, int64_t* out, int32_t n) {
  if (!prog || !out) return fail(WFM_EINVAL, "null program or output");
  const int64_t v[8] = {prog->dev.tile_samples, prog->dev.pkt_cap, prog->dev.n_slots, prog->n_tiles,
                        (int64_t)prog->packets.bytes, (int64_t)(prog->arena.bytes + prog->tile_tables.bytes), prog->dev.unit,
                        (int64_t)wfm::sample_smem_bytes(prog->dev, WFM_F64, false)};
  for (int i = 0; i < n && i < 8; ++i) out[i] = v[i];
  return WFM_OK;
}

static int check_launch(wfm_program_t prog, const WfmLaunch* l, int64_t* first, int64_t* count, int64_t* need) {
  if (!prog || !l) return fail(WFM_EINVAL, "null program or launch");
  const int64_t nw = (int64_t)prog->waves.size();
  *first = l->first_wave;
  *count = l->n_wave == 0 ? nw - l->first_wave : l->n_wave;
  if (*first < 0 || *count < 0 || *first + *count > nw) return fail(WFM_EINVAL, "channel range out of bounds");
  if (l->dtype != WFM_F64 && l->dtype != WFM_F32 && l->dtype != WFM_F32_FAST && l->dtype != WFM_C128 && l->dtype != WFM_I16)
    return fail(WFM_EINVAL, "bad dtype");
  if (prog->any_complex && l->dtype != WFM_C128)
    for (int64_t w = *first; w < *first + *count; ++w)
      if (prog->waves[w].flags & WFM_WAVE_COMPLEX)
        return fail(WFM_EINVAL, "channel %lld has complex amplitudes: request WFM_C128 output", (long long)w);
  if (prog->windowed && (l->dtype == WFM_C128 || l->accumulate))
    return fail(WFM_EUNSUPPORTED, "a windowed program writes real samples only: no WFM_C128 output, no accumulate");
  int64_t lo, ext;
  output_extent(prog, *first, *count, &lo, &ext);
  *need = ext;
  if (!l->out && ext > 0) return fail(WFM_EINVAL, "null output buffer");
  if (l->out_elems < ext) return fail(WFM_EINVAL, "output buffer too small: %lld < %lld", (long long)l->out_elems, (long long)ext);
  return WFM_OK;
}

// the launch(es) of one sampling request: channels [first, first + count) -> out (device)
static int launch_request(wfm_program_t prog, int64_t first, int64_t count, int dtype, int accumulate, void* out,
                          cudaStream_t st, const double* quant = nullptr) {
  const int64_t t0 = prog->tile_prefix[first], t1 = prog->tile_prefix[first + count];
  if (dtype != WFM_C128) {
    WFM_CUDA(wfm::launch_sample(prog->dev, prog->d_tiles, t0, t1 - t0, dtype, accumulate, out, st, quant));
    return WFM_OK;
  }
  // complex128: real and imaginary plane by the real-valued kernel into scratch, then
  // interleaved.  The scratch belongs to the program: complex launches of one program must be
  // stream-ordered.
  const int64_t total = (prog->total_samples + 3) & ~(int64_t)3, nw = (int64_t)prog->waves.size();  // plane stride
  const size_t bytes = sizeof(double) * (size_t)std::max<int64_t>(total, 4) * 2;
  if (prog->cscratch.bytes < bytes) {
    pool::release(prog->device, prog->cscratch);
    prog->cscratch = pool::Block{nullptr, 0};
    cudaError_t ea = pool::alloc(prog->device, bytes, &prog->cscratch);
    if (ea != cudaSuccess)
      return fail(WFM_ENOMEM, "allocating the %zu-byte plane scratch failed: %s", bytes, cudaGetErrorString(ea));
  }
  double* re = (double*)prog->cscratch.p;
  double* im = nullptr;
  if (prog->planar) {
    WfmProgram* q = prog->planar;
    im = re + total;
    const int64_t a0 = q->tile_prefix[first], a1 = q->tile_prefix[first + count];
    const int64_t b0 = q->tile_prefix[nw + first], b1 = q->tile_prefix[nw + first + count];
    WFM_CUDA(wfm::launch_sample(q->dev, q->d_tiles, a0, a1 - a0, WFM_F64, 0, re, st));
    WFM_CUDA(wfm::launch_sample(q->dev, q->d_tiles, b0, b1 - b0, WFM_F64, 0, re, st));
  } else {
    WFM_CUDA(wfm::launch_sample(prog->dev, prog->d_tiles, t0, t1 - t0, WFM_F64, 0, re, st));
  }
  WFM_CUDA(wfm::launch_interleave_c128(prog->d_tiles + t0, t1 - t0, prog->dev.waves, prog->dev.planes == 2, re, im, out,
                                       accumulate, st));
  return WFM_OK;
}

// the WFM_I16 requirements of a launch (wfm_sample_quant / wfm_sample_quant_host), after check_launch
static int check_quant(wfm_program_t prog, const WfmLaunch* l, const WfmQuant* q) {
  if (l->dtype != WFM_I16) return fail(WFM_EINVAL, "wfm_sample_quant writes WFM_I16 codes only (dtype %d)", l->dtype);
  if (l->accumulate) return fail(WFM_EINVAL, "DAC codes cannot be accumulated");
  if (!q || !q->row_gain_offset) return fail(WFM_EINVAL, "null gain / offset table");
  if (!prog->rows_aligned8)
    return fail(WFM_EINVAL, "WFM_I16 output needs every row at a multiple of 8 samples (lower the batch with align=8)");
  return WFM_OK;
}

static int sample_device(wfm_program_t prog, const WfmLaunch* l, const double* quant, void* stream, int64_t first,
                         int64_t count) {
  if ((uintptr_t)l->out % 16) return fail(WFM_EINVAL, "output buffer must be 16-byte aligned");
  DeviceGuard g(prog->device);
  const int64_t t0 = prog->tile_prefix[first], t1 = prog->tile_prefix[first + count];
  int rc = launch_request(prog, first, count, l->dtype, l->accumulate, l->out, (cudaStream_t)stream, quant);
  if (rc != WFM_OK) return rc;
  if (t1 > t0) {
    prog->launches += 1;
    std::lock_guard<std::mutex> lk(prog->ev_mu);
    cudaEvent_t ev = nullptr;
    for (auto& se : prog->launch_events)
      if (se.first == (cudaStream_t)stream) ev = se.second;
    if (!ev) {
      WFM_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      prog->launch_events.emplace_back((cudaStream_t)stream, ev);
    }
    WFM_CUDA(cudaEventRecord(ev, (cudaStream_t)stream));
  }
  return WFM_OK;
}

int wfm_sample(wfm_program_t prog, const WfmLaunch* l, void* stream) {
  int64_t first, count, need;
  int rc = check_launch(prog, l, &first, &count, &need);
  if (rc != WFM_OK) return rc;
  if (l->dtype == WFM_I16) return fail(WFM_EINVAL, "WFM_I16 output takes a gain / offset table: call wfm_sample_quant");
  return sample_device(prog, l, nullptr, stream, first, count);
}

int wfm_sample_quant(wfm_program_t prog, const WfmLaunch* l, const WfmQuant* q, void* stream) {
  int64_t first, count, need;
  int rc = check_launch(prog, l, &first, &count, &need);
  if (rc == WFM_OK) rc = check_quant(prog, l, q);
  if (rc != WFM_OK) return rc;
  return sample_device(prog, l, q->row_gain_offset, stream, first, count);
}

static int sample_host(wfm_program_t prog, const WfmLaunch* l, const double* quant, int64_t first, int64_t count,
                       int64_t need) {
  if (l->accumulate) return fail(WFM_EUNSUPPORTED, "accumulate is not available with host buffers");
  StageTimer tm("sample_host");
  const cudaStream_t ST = cudaStreamPerThread;  // see wfm_program_create
  DeviceGuard g(prog->device);
  const size_t esz = l->dtype == WFM_F64 ? 8 : ((l->dtype == WFM_F32 || l->dtype == WFM_F32_FAST) ? 4 : (l->dtype == WFM_I16 ? 2 : 16));
  // only the extent actually covered by the requested channels is staged/copied
  int64_t lo, hi;
  output_extent(prog, first, count, &lo, &hi);
  if (count == 0 || need == 0) return WFM_OK;
  const size_t bytes = (size_t)need * esz;
  if (prog->stage.bytes < bytes) {
    pool::release(prog->device, prog->stage);
    prog->stage = pool::Block{nullptr, 0};
    cudaError_t ea = pool::alloc(prog->device, bytes, &prog->stage);
    if (ea != cudaSuccess) return fail(WFM_ENOMEM, "allocating the %zu-byte staging buffer failed: %s", bytes, cudaGetErrorString(ea));
  }
  tm.lap("stage alloc");
  // padding between channels is never written by the kernel: keep it defined (nothing to do when the rows are gapless)
  if (!(prog->gapless && first == 0 && count == (int64_t)prog->waves.size())) WFM_CUDA(cudaMemsetAsync((char*)prog->stage.p + (size_t)lo * esz, 0, (size_t)(need - lo) * esz, ST));
  const int64_t t0 = prog->tile_prefix[first], t1 = prog->tile_prefix[first + count];
  {
    const int rc2 = launch_request(prog, first, count, l->dtype, 0, prog->stage.p, ST, quant);
    if (rc2 != WFM_OK) return rc2;
  }
  if (t1 > t0) prog->launches += 1;
  WFM_CUDA(cudaMemcpyAsync((char*)l->out + (size_t)lo * esz, (char*)prog->stage.p + (size_t)lo * esz,
                           (size_t)(need - lo) * esz, cudaMemcpyDeviceToHost, ST));
  // A long copy is waited for on a blocking-sync event: the host thread sleeps instead of spinning on the stream for
  // hundreds of milliseconds (one process per GPU with two submitting threads each is more threads than an 8-GPU host
  // has cores to spin on).  Short copies keep the spinning wait: its wake-up is tens of microseconds faster.
  if ((size_t)(need - lo) * esz >= kBlockingWaitBytes) {
    static thread_local cudaEvent_t ev[pool::kMaxDevices] = {};
    const int dv = prog->device;
    if (dv >= 0 && dv < pool::kMaxDevices) {
      if (!ev[dv]) WFM_CUDA(cudaEventCreateWithFlags(&ev[dv], cudaEventBlockingSync | cudaEventDisableTiming));
      WFM_CUDA(cudaEventRecord(ev[dv], ST));
      WFM_CUDA(cudaEventSynchronize(ev[dv]));
    } else {
      WFM_CUDA(cudaStreamSynchronize(ST));
    }
  } else {
    WFM_CUDA(cudaStreamSynchronize(ST));
  }
  tm.lap("memset+kernel+D2H");
  return WFM_OK;
}

int wfm_sample_host(wfm_program_t prog, const WfmLaunch* l) {
  int64_t first, count, need;
  int rc = check_launch(prog, l, &first, &count, &need);
  if (rc != WFM_OK) return rc;
  if (l->dtype == WFM_I16) return fail(WFM_EINVAL, "WFM_I16 output takes a gain / offset table: call wfm_sample_quant_host");
  return sample_host(prog, l, nullptr, first, count, need);
}

int wfm_sample_quant_host(wfm_program_t prog, const WfmLaunch* l, const WfmQuant* q) {
  int64_t first, count, need;
  int rc = check_launch(prog, l, &first, &count, &need);
  if (rc == WFM_OK) rc = check_quant(prog, l, q);
  if (rc != WFM_OK) return rc;
  return sample_host(prog, l, q->row_gain_offset, first, count, need);
}

int wfm_quantize(const double* x, int16_t* y, int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                 const double* gain_offset, void* stream) {
  if (n_sig < 0 || n < 0) return fail(WFM_EINVAL, "negative size");
  if (n_sig == 0 || n == 0) return WFM_OK;
  if (!x || !y || !gain_offset) return fail(WFM_EINVAL, "null pointer");
  if (n_sig > 1 && (x_stride < n || y_stride < n)) return fail(WFM_EINVAL, "row stride smaller than the row");
  WFM_CUDA(wfm::launch_quantize(x, y, n_sig, n, x_stride, y_stride, gain_offset, (cudaStream_t)stream));
  return WFM_OK;
}

}  // extern "C"
