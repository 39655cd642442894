// wfm_internal.h — structures shared by the C-ABI layer and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/wfm_b200.h"

namespace wfm {

// samples per tile of the sampling kernel.  A tile is assembled by ONE WARP in its
// private slice of shared memory (tile_samples x 8 B) and stored with one TMA bulk
// copy.  Chosen per program from the table density: dense programs take smaller
// tiles so that the tile's packet fits the warp's slice.
constexpr int kMinBlocks = 2;  // resident 8-warp CTAs per SM the kernel is sized for
constexpr int kWarps = 8;      // autonomous warps per CTA
// Samples one lane evaluates together (a UNIT: consecutive samples of one active segment),
// chosen per program (DevProgram::unit).  Two samples per lane run as independent dependency
// chains and pay the row decoding once: the dense case (RB batches: every sample active,
// many rounds per tile; +39 % measured on cfg3).  One sample per lane needs fewer registers
// and half the slot memory: the sparse case (control frames: at most ~2 rounds per tile;
// +4.5 % measured on cfg2).
constexpr int kMinTileSamples = 128;
constexpr int kMaxTileSamples = 1536;
// shared memory per warp: 8 * kMinBlocks warps share the SM's 227 KB (1 KB per CTA is reserved by the
// driver).  The erf coefficient table is read through L1: a shared-memory copy per CTA (2.5 KB) was
// measured within noise of it (610 vs 616 GSa/s on cfg2), so the shared memory goes to the packet buffers.
constexpr int kWarpSliceBytes = ((227 * 1024 / kMinBlocks - 1024) / kWarps) & ~127;

// The DENSE kernel (programs whose samples are mostly active, e.g. randomized-benchmarking batches): one CTA of 12
// autonomous warps per SM at up to 168 registers, four samples per lane unit, results stored straight from registers
// (no tile buffer): its warp slice holds the value slots and the two packet buffers only.
constexpr int kDenseWarps = 12;
constexpr int kDenseUnit = 4;
constexpr int kDenseSliceBytes = ((227 * 1024 - 1024) / kDenseWarps) & ~127;

// Value slots of one segment evaluation: per lane kMaxSlots + 1 slots of `unit`
// doubles in the warp's shared slice, slot-major (slot k of lane l at byte
// k * slot_stride(unit) + l * 8 * unit: conflict-free).  Slot 0 always holds 1.0.
constexpr int kMaxSlots = 12;
__host__ __device__ constexpr int slot_stride(int unit) { return 32 * 8 * unit; }  // bytes between consecutive slots

// One warp's slice of the sampling kernels' dynamic shared memory (every part 16-byte aligned):
//   [tile buffers: planes x tile_samples x element][value slots: n_slots x slot_stride(unit)][packet buffer 0]
//   [packet buffer 1][2 mbarriers]
// planes = 2 when the program holds I/Q pairs (one tile buffer per output row); the dense kernel keeps none (0).
struct WarpSlice {
  size_t tile_bytes, slot_bytes, pkt_cap;
  __host__ __device__ size_t slots() const { return tile_bytes; }
  __host__ __device__ size_t packets() const { return tile_bytes + slot_bytes; }
  __host__ __device__ size_t barriers() const { return packets() + 2 * pkt_cap; }
  __host__ __device__ size_t bytes() const { return (barriers() + 16 + 127) & ~(size_t)127; }
  // the largest packet buffer (16-byte multiple) whose slice fits `budget` bytes; may be negative
  int max_pkt_cap(int budget) const { return ((budget - (int)tile_bytes - ((int)slot_bytes + 16 + 128)) / 2) & ~15; }
};
__host__ __device__ inline WarpSlice warp_slice(int planes, int tile_samples, int elem_bytes, int n_slots, int unit, int pkt_cap) {
  return WarpSlice{(size_t)planes * tile_samples * elem_bytes, (size_t)n_slots * slot_stride(unit), (size_t)pkt_cap};
}

// ---- the device program of ONE active segment (built on the device at upload) ------------
// The ABI factor rows of a segment are regrouped so that the interpreter decodes no opcode
// on the hot rows and never stores a sine:
//   per WFM_COS_SINCOS row, in ABI order:
//     SRow          slot <- cos(a), a = w * (x - shift); (cos a, sin a) stay in registers for
//     CRow[n_child] slot <- cos(w * (x - shift')) of every WFM_COS_ROT row based on it, by rotation
//   GRow[n_gen]     everything else (switch on the basis id)
//   CTerm[n_term]
// Value slots follow that order (slot 0 holds 1.0): one per SRow, CRow and GRow.  The ABI's
// WFM_NOP rows (sine placeholders) vanish.
struct SRow {
  double shift, w;
  uint32_t n_child;  // CRows that follow
  uint32_t pad0;
  // two-sample units on an affine grid: the second sample's (cos, sin) by rotation of the
  // first's by D = w * delta (+ the measured residual), instead of a second range reduction
  double D, cD, sD;
};
static_assert(sizeof(SRow) == 48, "SRow layout");

// cos(a_t), a_t = w * (x - shift) rounded exactly as the reference rounds it, from the parent's
// (cos, sin)(a): a_t = a + D + eps with D ~ w * (parent shift - shift) a host constant (cos D,
// sin D tabulated) and eps = (a_t - a) - D the MEASURED residual (|eps| ~ ulp(a))
struct CRow {
  double shift;
  double D, cD, sD;
};
static_assert(sizeof(CRow) == 32, "CRow layout");

struct GRow {
  int32_t func;     // WFM_* basis id
  int32_t arg_off;  // its block in the argument pool (global memory)
  double shift, a0, a1;
};
static_assert(sizeof(GRow) == 32, "GRow layout");

// amp * v[o0] * v[o1] * v[o2]: up to three exponent-1 references as BYTE offsets of
// their value slots for unit = 1 (slot * 256; the kernel scales them by its unit); a
// missing reference points at slot 0 (1.0; x * 1.0 is exact),
// so the product needs no loop and no branch.  Terms that do not fit (more
// references, an exponent != 1) carry kCTermExt and are read from the ABI tables.
struct CTerm {
  double amp;
  uint16_t o0, o1, o2;
  uint16_t flags;
};
static_assert(sizeof(CTerm) == 16, "CTerm layout");
constexpr uint32_t kCTermGroupEnd = 1, kCTermExt = 2;
// first term of the SECOND row of an I/Q pair: the first row's sum is complete (stored before this term is added)
constexpr uint32_t kCTermPlaneSwitch = 4;

// per segment, parallel to the ABI segment table
struct SegPlan {
  uint8_t n_sc, n_rot, n_gen, flags;  // n_rot: CRows of all SRows together
  uint16_t n_term;
  uint16_t blk16;  // bytes / 16 of its rows + terms in a packet (0 for a wide segment)
};
static_assert(sizeof(SegPlan) == 8, "SegPlan layout");
// more value slots / terms than the hot path holds: evaluated row by row from the ABI tables
constexpr uint32_t kSegWide = 1;

// ---- tile packets: the device IR the sampling kernel executes ------------------------------
// Built once per program on the device.  A packet is everything ONE tile needs,
// contiguous in global memory (16-byte aligned, size a multiple of 16) so that a
// warp brings it into shared memory with ONE TMA bulk copy:
//   PacketHeader | ARow[n_arows + 1] | PatchRow[n_patch] | per active segment: {SRow CRow..}.. GRow.. CTerm..
// Zero segments do not appear at all: the kernel fills the tile with `base` first.
struct PacketHeader {
  int64_t out0;   // index of the tile's first sample in the output buffer
  int64_t j0;     // first sample of the tile in its channel
  double base;    // value of the channel's zero segments (its accumulator start)
  double t0, delta;  // affine grid of the channel: x[j] = t0 + j*delta
  int32_t wave;
  uint32_t flags;    // WfmWave::flags | kPacketCold
  uint16_t cnt;      // samples in the tile
  uint16_t n_arows;  // active segments intersecting the tile
  uint16_t n_patch;  // flat segments whose value differs from `base`
  uint16_t n_units;  // units (DevProgram::unit consecutive samples of one active segment) in the tile
  uint32_t reserved[2];
  int64_t out1;   // WFM_WAVE_PAIR: the same tile of the second row
  double base1;   //                and that row's zero-segment value
};
static_assert(sizeof(PacketHeader) == 80, "PacketHeader layout");
constexpr uint32_t kPacketCold = 0x80000000u;  // header only: the tile takes the global-table path

// one ACTIVE segment of the tile; row n_arows is a sentinel closing the ranges
struct ARow {
  uint16_t start;  // first tile-sample of the segment
  uint16_t first;  // units of the tile before this segment
  uint16_t rel;    // bits 0..11: offset / 16 of its rows within the packet; bits 12..15: SegPlan flags
  uint16_t len;    // its samples inside the tile
  uint8_t n_sc, n_rot, n_gen, n_term;
  int32_t gseg;    // absolute segment row (extended terms, wide segments)
};
static_assert(sizeof(ARow) == 16, "ARow layout");

// a flat run [a, b) of the tile with its own value
struct PatchRow {
  uint16_t a, b;
  uint32_t plane;  // 0 / 1: row of an I/Q pair
  double val;
};
static_assert(sizeof(PatchRow) == 16, "PatchRow layout");

// device-resident copy of a lowered batch (all DEVICE pointers)
struct DevProgram {
  const WfmWave* waves;
  const double* seg_bound;
  const WfmSegPtr* seg_ptr;
  const WfmFactor* facs;   // ABI rows
  const WfmTerm* terms;
  const WfmRef* refs;
  const double* args;
  const double* x;
  // built on the device once per program (prepare kernels):
  const SegPlan* seg_plan;   // [n_segs]
  const uint8_t* row_slot;   // [n_facs] value slot of every ABI factor row (0 for WFM_NOP rows)
  const CTerm* cterms;       // parallel to terms
  const int32_t* seg_start;  // [n_segs] first sample (channel-relative) owned by the segment
  const double* seg_val;     // [n_segs] value of a FLAT segment (offset + constant terms, clipped)
  const double* seg_val1;    // [n_segs] the same for the second row of I/Q pairs (planes == 2)
  const int32_t* seg_wave;   // [n_segs] owning channel (host-built; pre-pass only)
  const uint32_t* pkt_off;       // [n_tiles + 1] packet offsets in 16-byte units
  const unsigned char* packets;  // the tile packets
  int unit;          // samples per lane unit: 1 or 2 (sparse kernel), kDenseUnit = 4 (dense kernel)
  int tile_samples;  // kMinTileSamples .. kMaxTileSamples, multiple of 128
  int n_slots;       // value slots per lane in shared memory: 1 (the constant 1.0) + max rows per segment
  int pkt_cap;       // bytes of ONE packet buffer in a warp's shared slice (two buffers per warp)
  int planes;        // 2 if any channel is an I/Q pair (two tile buffers per warp), else 1
  int dense;         // 1: sampled by the dense kernel (unit == kDenseUnit, every flat segment listed as a patch row)
};

// one warp's work item: up to DevProgram::tile_samples consecutive samples of channel `wave`
struct TileDesc {
  int64_t j0;    // first sample of the tile in its channel
  int64_t out0;  // index of that sample in the output buffer
  int32_t wave;
  int32_t cnt;   // samples in the tile
  // filled on the device by prepare_tiles_kernel (once per program):
  int32_t seg0;  // ABSOLUTE segment row that owns the tile's first sample
  int32_t nb;    // segment rows the tile spans
};
static_assert(sizeof(TileDesc) == 32, "TileDesc layout");

struct PrepareCounts {
  int64_t n_waves, n_segs, n_facs, n_terms, n_tiles;
  int64_t n_windows;  // windowed program (wfm_program_create_windows): tiles per window; 0: tiles per channel
};

// tables the pre-pass writes (device pointers into the program's arena)
struct PrepareBuffers {
  int32_t* seg_wave;
  int32_t* seg_start;
  double* seg_val;
  double* seg_val1;
  SegPlan* seg_plan;
  uint8_t* row_slot;
  CTerm* cterms;
  TileDesc* tiles;
  const WfmWindow* windows;    // [n_windows] (windowed programs; NULL otherwise)
  const int64_t* tile_prefix;  // [n_waves + 1] tiles before channel w, or [n_windows + 1] before window w (host-built)
  uint32_t* pkt_size;          // [n_tiles + 1]
};

// pass 1a: owning channel of every segment, segment start positions, flat values, segment
// plans, slot map, compact terms (independent of the tile size)
cudaError_t launch_prepare_segments(const DevProgram& P, const PrepareCounts& n, const PrepareBuffers& b, cudaStream_t stream);
// total[0] += samples owned by active segments (needs seg_start; decides DevProgram::unit)
cudaError_t launch_count_active(const DevProgram& P, int64_t n_segs, unsigned long long* total, cudaStream_t stream);
// pass 1b: the tile rows with their segment range and packet size (16-byte units) ->
// tiles[n_tiles], pkt_size[n_tiles] (either may be NULL: sizing pass) and, if stats != NULL,
// stats[0] = max packet size (16-byte units, as if every packet fitted), stats[1] = tiles that do not fit P.pkt_cap
cudaError_t launch_prepare_tiles(const DevProgram& P, const PrepareCounts& n, const PrepareBuffers& b, uint32_t* stats,
                                 cudaStream_t stream);
// exclusive scan: pkt_size[n] -> pkt_off[n + 1] (pkt_off[n] = total); scratch holds ceil(n / 4096) + 1 words
cudaError_t launch_scan(const uint32_t* pkt_size, uint32_t* pkt_off, uint32_t* scratch, int64_t n, cudaStream_t stream);
// pass 2: write the packets (windowed programs: b.windows / b.tile_prefix give a pair tile's second row)
cudaError_t launch_fill_packets(const DevProgram& P, const TileDesc* tiles, int64_t n_tiles, const PrepareCounts& n,
                                const PrepareBuffers& b, unsigned char* packets, cudaStream_t stream);
// a warp's shared-memory slice for the program's kernel, with tiles of tile_samples elements of elem_bytes
inline WarpSlice program_slice(const DevProgram& P, int tile_samples, int elem_bytes, int pkt_cap) {
  if (P.dense) return warp_slice(0, 0, 0, P.n_slots, kDenseUnit, pkt_cap);
  return warp_slice(P.planes == 2 ? 2 : 1, tile_samples, elem_bytes, P.n_slots, P.unit, pkt_cap);
}
// the packet buffer capacity of tiles of tile_samples: the largest that fits the kernel's warp slice when the
// tile buffers hold fp64 (fp32 and int16 output use a smaller slice with the same buffers, fp32 accumulate this one)
inline int packet_capacity(const DevProgram& P, int tile_samples) {
  return program_slice(P, tile_samples, 8, 0).max_pkt_cap(P.dense ? kDenseSliceBytes : kWarpSliceBytes);
}
// dynamic shared memory of a sampling launch (accumulate: fp64 tile buffers whatever the output type)
size_t sample_smem_bytes(const DevProgram& P, int dtype, bool accumulate);

// quant: WFM_I16 only, the DEVICE [n_waves][2][2] (gain, offset) table of WfmQuant
cudaError_t launch_sample(const DevProgram& P, const TileDesc* tiles, int64_t tile_begin, int64_t n_tiles, int dtype,
                          int accumulate, void* out, cudaStream_t stream, const double* quant = nullptr);
// y[s][j] = dac_code(x[s][j], gain_offset[s][0], gain_offset[s][1])
cudaError_t launch_quantize(const double* x, int16_t* y, int64_t n_sig, int64_t n, int64_t x_stride, int64_t y_stride,
                            const double* gain_offset, cudaStream_t stream);
// out[tile samples] = (re, im) (+ out when accumulate), and the same for the second row of the tiles of I/Q pairs
// (pairs: the program holds any, waves: its DEVICE channel table); im may be NULL (zero imaginary part)
cudaError_t launch_interleave_c128(const TileDesc* tiles, int64_t n_tiles, const WfmWave* waves, bool pairs, const double* re,
                                   const double* im, void* out, int accumulate, cudaStream_t stream);

}  // namespace wfm
