// ilf_common.cuh -- shared device-side definitions of libilf_b200 (sm_100a).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <mutex>

#include "ilf_b200.h"

namespace ilf {

// Geometry shared by every slot of a context; passed to kernels by value.
struct Geom {
  int width, height;        // luma samples
  int pitch_y, pitch_c;     // plane pitches in samples (multiples of 64 -> 128-byte rows)
  int units_w, units_h;     // 4x4 luma units
  int units_pitch;          // row pitch of the device-side unit grids (units_w rounded up to 4: TMA rows are multiples of 16 bytes)
  int ctu_log2, ctus_w, ctus_h;
  int bd_luma, bd_chroma;
  // Band mode (one picture split into CTU-row bands across GPUs): the slot's planes hold picture rows
  // [row0, row0 + rows) of the full picture; filtering decisions use full-picture coordinates.
  int row0, rows;           // luma rows held (row0 multiple of 8); whole picture: 0, height
  int out_row0, out_rows;   // luma rows this context must produce (its own CTU rows)
  int debug;                // measurement aid (env ILF_DEBUG): bit 0 = kernels stage and write back only (no filtering)
};

// Per-slot device pointers; an array of these lives in device memory (one entry per slot) and kernels index
// it with first_slot + blockIdx.z, so one launch covers a batch of pictures.
// Tile geometry of the band-walking kernels (ilf_ring.cuh): the TMA box sizes are baked into the tensor maps that
// ilf_create encodes, so they live here.
constexpr int RING_TILE_W = 128;   // samples per tile row, all planes (256-byte box rows)
// The ALF kernels walk narrower tiles: 64 samples, 128-thread CTAs, five per SM, each with its own ring and barriers -- the
// phases of more, smaller CTAs interleave better than those of three 256-thread CTAs (0.420 vs 0.447 ms for 17 4K pictures).
// Their TMA boxes are ALF_TILE_W + 16 wide.
#ifndef ALF_TILE_W
#define ALF_TILE_W 64
#endif
constexpr int ALF_TILE = ALF_TILE_W;
#ifndef SAO_TILE_W
#define SAO_TILE_W 128
#endif
constexpr int SAO_TILE = SAO_TILE_W;   // tile width of the SAO walk (its TMA boxes are SAO_TILE x 34)
constexpr int DB_BAND_ROWS = 32;   // luma rows a deblocking CTA owns (shifted up by 4 rows; chroma: 16 rows shifted by 2)
// Deblocking works on independent tiles: a box carries the tile plus the reach of the vertical edges on its borders (4 luma / 2
// chroma samples, 1 unit), widened to 8 samples / 4 units on each side because a TMA box must START on a 16-byte boundary
// (a box that starts 8 bytes off faults with "illegal instruction"); motion boxes start 2 (int16: 8 bytes per unit) / 1 (int32)
// units left of the tile and are counted in 32-bit words (2 / 4 per unit; rows are multiples of 16 bytes).
constexpr int DB_BOX_W = RING_TILE_W + 16, DB_BOX_CW = RING_TILE_W / 2 + 16, DB_BOX_UNITS = RING_TILE_W / 4 + 8;
constexpr int DB_BOX_MV16_WORDS = (RING_TILE_W / 4 + 4) * 2, DB_BOX_MV32_WORDS = (RING_TILE_W / 4 + 2) * 4;
constexpr int SAO_BAND_ROWS = 32;  // rows a SAO CTA owns; the box adds one halo row above and below
constexpr int ALF_BAND_ROWS = 32;  // rows an ALF CTA owns; the box adds 3 (luma, 7x7 + classification) or 2 (chroma, 5x5) halo rows on each side
constexpr int ALF_HALO_Y = 3, ALF_HALO_C = 2;

struct alignas(64) SlotDev {
  // TMA descriptors of the slot's planes, tensor (x, y, buffer): dims (plane width, held rows, 3)
  CUtensorMap tm_db[3];     // box DB_BOX_W x DB_BAND_ROWS (luma), DB_BOX_CW x DB_BAND_ROWS/2 (chroma)
  CUtensorMap tm_info, tm_info_c;  // unit grids, tensor (unit x, unit y, 1) of uint32: box DB_BOX_UNITS x 8
  CUtensorMap tm_mv16, tm_mv32;    // motion vectors as uint32 words (2 / 4 per unit): box DB_BOX_MV16_WORDS x 8 / DB_BOX_MV32_WORDS x 8
  CUtensorMap tm_sao[3];    // box SAO_TILE x (SAO_BAND_ROWS + 2)
  CUtensorMap tm_alf[3];    // box (ALF_TILE + 16) x (ALF_BAND_ROWS + 2 * halo), loaded 8 samples left of the tile
  int16_t* buf[3][3];       // [buffer: 0 = input, 1, 2 = work][plane]
  const uint32_t* info;     // deblock grid, luma tree
  const uint32_t* info_c;   // chroma tree layer or nullptr
  const int16_t* mv16;
  const int32_t* mv32;
  const uint8_t* ctu_slice;
  const ilf_deblock_params* db_params;
  const ilf_sao_ctu* sao;
  const ilf_alf_params* alf;
  const int* alf_coef;            // [25 classes][4 transposes][16] luma coefficients, transposition applied (set by ilf_set_alf_params)
  const uint32_t* alf_coef_dp;    // [25][4][20] the same filters in the dot-product layout (ilf_alf_tab.cuh), then [16] words of the chroma filter
  int alf_mode;                   // bit 0 / 1: the luma filters / the chroma filter fit the dot-product path (else the general path);
                                  // bit 2 / 3: only their centre coefficient has a high part
  const uint8_t* alf_ctu_enable;  // [3][num_ctus]
  uint8_t* alf_class;             // [units_h][units_w] scratch / output of ilf_alf_classify
  const int16_t* org[3];          // source picture of the encoder (ilf_set_original), plane pitches as buf
  const uint8_t* stats_avail;     // [num_ctus] ILF_AVAIL_* of the statistics pass
  long long* stats;               // [num_ctus][3][5][64] SAO statistics (ilf_sao_stats)
  long long* alf_stats;           // [num_ctus][ILF_ALF_STATS_WORDS] ALF statistics (ilf_alf_stats)
};

// Per-launch control word of every slot of a batch (kernel parameter, indexed with blockIdx.z).  Each plane of a
// slot lives in one of the slot's three buffers; a stage reads plane p from buffer src_p and writes the other work
// buffer (dst = src == 1 ? 2 : 1, never buffer 0 = the uploaded input).  A plane whose stage is off for the whole
// picture (the reference returns early: SampleAdaptiveOffset.cpp:572-583, AdaptiveLoopFilter.cpp:70-73) is skipped:
// no CTA touches it and its result stays where it was.
constexpr int MAX_BATCH = 128;
struct BatchCtl {
  uint16_t v[MAX_BATCH];     // bits 2p..2p+1: source buffer of plane p; bit 6+p: skip plane p; bits 9..13: CTL_ALF_*
  uint8_t slot[MAX_BATCH];   // slot (relative to first_slot) that grid layer blockIdx.z works on: launches cover active slots only
};
// ALF launches: arithmetic path and luma filter shape of the slot (ilf_set_alf_params), so that a CTA knows them without a load
constexpr unsigned CTL_ALF_DOT_Y = 1u << 9, CTL_ALF_7X7 = 1u << 10, CTL_ALF_HIC_Y = 1u << 11, CTL_ALF_DOT_C = 1u << 12, CTL_ALF_HIC_C = 1u << 13;
__host__ __device__ __forceinline__ int ctl_src(unsigned c, int plane) { return (c >> (2 * plane)) & 3; }
__host__ __device__ __forceinline__ int ctl_dst(unsigned c, int plane) { return ctl_src(c, plane) == 1 ? 2 : 1; }
__host__ __device__ __forceinline__ bool ctl_skip(unsigned c, int plane) { return (c >> (6 + plane)) & 1; }

__device__ __forceinline__ int clip3i(int lo, int hi, int v) { return min(max(v, lo), hi); }

// 128-bit / 64-bit global accesses.  Pictures are streamed once per stage: bypass L1 allocation on loads
// that have no intra-CTA reuse.
__device__ __forceinline__ uint2 ldg_u2(const void* p) { return __ldg(reinterpret_cast<const uint2*>(p)); }
__device__ __forceinline__ uint4 ldg_u4(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// Band-walking launches: a band (one CTA walking `ntx` tiles) can be cut into `nseg` horizontal segments so that a small batch
// still fills the machine.  Picks the nseg whose CTA count comes closest to a whole number of waves of `resident` CTAs
// (a partly filled last wave is idle hardware), discounted by the ring's start-up cost for short segments.
inline int pick_segments(int bands_total, int ntx, int resident, float startup_tiles = 0.5f) {
  int best = 1;
  float best_score = -1.f;
  for (int nseg = 1; nseg <= ntx; nseg++) {
    const float len = (float)ntx / nseg;
    if (nseg > 1 && len < 2.f) break;
    const float waves = (float)bands_total * nseg / resident;
    const float eff = waves / (float)(int)(waves + 0.999f);
    const float score = eff * len / (len + startup_tiles);
    if (score > best_score * 1.02f) { best_score = score; best = nseg; }  // prefer fewer, longer segments unless clearly better
  }
  return best;
}

// Experiment knob: extra dynamic shared memory per CTA (bytes, from the environment) -- caps how many CTAs of a kernel an SM holds,
// which is how mixed residency of two kernels running on different streams is steered (tools/exp_lanes.py).
inline int env_int(const char* name, int dflt = 0) { const char* v = getenv(name); return v ? atoi(v) : dflt; }

// cudaFuncSetAttribute is per device: a process may hold contexts on several GPUs (and threads), so "already raised" is tracked
// per device under a lock, and the caller raises the attributes while it holds it (set_attrs runs once per device).
template <typename F>
inline void once_per_device(bool (&seen)[64], F set_attrs) {
  static std::mutex mu;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return;
  std::lock_guard<std::mutex> lock(mu);
  if (seen[dev]) return;
  set_attrs();
  seen[dev] = true;
}

// Programmatic dependent launch: the stages of a chain are consecutive kernels on one stream.  Every kernel lets its
// successor be scheduled as soon as all of its own CTAs have started (pdl_launch_dependents, first instruction), and waits
// for its predecessor to have completed and flushed (pdl_wait) before it touches picture planes -- its prologue (barrier
// initialisation, tables, descriptors) and the predecessor's last wave overlap.  ILF_NO_PDL=1 launches the plain way.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  static const bool plain = getenv("ILF_NO_PDL") && atoi(getenv("ILF_NO_PDL")) != 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = plain ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// One launch covers `num_slots` <= MAX_BATCH grid layers; layer z works on slot first_slot + ctl.slot[z] under control word ctl.v[z].
void launch_deblock(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, int mv_mode, int* work, cudaStream_t st);
// ilf_deblock_search: adds sum((D_k - O)^2 >> shift) of every candidate k and plane to out[(first_slot + ctl.slot[z]) * 192 + 3 k + plane].
void launch_deblock_search(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, int mv_mode, const ilf_deblock_candidate* cands,
                           int num_cands, int shift_luma, int shift_chroma, unsigned long long* out, cudaStream_t st);
void launch_sao(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st);
void launch_alf(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, int planes /* bit 0 luma, bit 1 chroma */, cudaStream_t st);
void launch_sao_stats(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st);
cudaError_t picture_hash(const Geom& g, const int16_t* const planes[3], uint32_t* scratch, cudaStream_t st, uint32_t out_crc[3], uint32_t out_sum[3]);
// The same kernels over luma rows [first, first + n) of the held planes (chroma halved), y0 = their first picture row: the CRC register
// contribution from a zero register and the checksum partial sum (ilf_picture_hash_band).  Synchronises `st`.
cudaError_t hash_rows(const Geom& g, const int16_t* const planes[3], uint32_t* scratch, cudaStream_t st, int first, int n, int y0, uint32_t reg[3], uint32_t sum[3]);
void launch_alf_stats(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st);
void launch_alf_classify(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st);

}  // namespace ilf
