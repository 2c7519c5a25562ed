// ilf_deblock.cu -- deblocking filter, both edge directions fused in one pass (sm_100a).
//
// Replaces LoopFilter::loopFilterPic (LoopFilter.cpp:149-230): "all vertical edges of the picture, then all
// horizontal edges".  Filtered edges lie on the 8x8 luma grid (:313-324), each reads 4 and writes 3 samples
// per side (:856-916), and the on/off + strong/weak decisions of a 4-line segment use lines 0 and 3 of that
// segment only (:640-671).  Vertically, a band of 32 luma rows shifted up by 4 rows is therefore dependency-closed for
// the horizontal edges in its middle once its vertical edges are done.  Horizontally a TILE of 128 output columns
// [x0, x0 + 128) is dependency-closed once it is given four more columns on each side: the vertical edges x0 + 8e, e = 0..16,
// read [x0 - 4, x0 + 132) and leave [x0, x0 + 128) final (edge 16 is the next tile's edge 0: both tiles compute it, each keeps
// its own side).
//
// Data movement: INDEPENDENT TILES drawn from a raster-order work queue.  The tiles of a launch are numbered in raster order
// inside a picture (tile of a band, band: rows [32 ty - 4, 32 ty + 28), chroma [16 ty - 2, 16 ty + 14), units [8 ty - 1, 8 ty + 7)),
// picture after picture; 148 x 6 CTAs draw tile numbers from one device counter (atomicAdd; the last CTA to leave resets it for
// the next launch on the stream) and each keeps a ring of DB_STAGES shared-memory stages: the TMA boxes of a tile -- luma 144 x 32
// from x0 - 8, Cb and Cr 80 x 16 from cx0 - 8, and the tile's edge records (ilf_common.cuh DB_REC_*: 24 x 8 + 32 x 4 uint16 for luma,
// 16 x 8 + 32 x 2 uint32 for chroma, 1.4 KB) -- land in one stage while the tile of the other stage is filtered.  Because the queue hands tiles out in
// raster order whatever the CTAs' relative progress, the CTAs resident at any moment cover a compact window of the picture.
// That order is what the memory system rewards (profiles/r02_ring_vs_copy.txt, tools/ubench/tma_ring.cu): the same boxes moved by
// persistent CTAs that each walk a band -- the design of round 1 -- copy at 4.7 TB/s, handed out in raster order 5.7 TB/s, because
// a band walk spreads the concurrent accesses over every row of every picture (one 256-byte piece per DRAM page at a time).
// Per tile:
//   1. vertical edges x0 + 8e, e = 0..16 (luma) / cx0 + 8k, k = 0..8 (chroma), in shared memory;
//   2. a CTA barrier;
//   3. horizontal edges: a task (4 luma columns x 8 rows, or 2 chroma columns x 8 rows) loads its block, filters the edge in its
//      middle when there is one, and stores the block straight to the destination plane: a warp's 32 tasks write 256 (128)
//      contiguous, sector-aligned bytes per row.  There is no separate write-back pass;
//   4. a CTA barrier, after which the stage is refilled with the tile drawn during step 3.
// Every sample crosses HBM once in and once out (the reference makes two picture passes); the 16 halo columns of a box are
// L2 hits (the neighbouring tiles are in flight at the same time).
//
// Edge records.  Everything about a segment that does not depend on the samples -- edge flag and bS (xGetBoundaryStrengthSingle
// :419-541), the no-filter sides, the QP with the slice's beta / tc offsets applied as table indices (:626-634), for chroma the
// plane's QP offset and mapping (:811-829) -- is fixed once the picture's side information is: deblock_records_kernel derives it
// from the packed per-4x4 grid and motion vectors (include/ilf_b200.h) when ilf_set_deblock_info copies them, on a stream of its own,
// into a 16-bit record per segment.  deblock_kernel reads the records instead of the grid and the motion vectors (about 1.4 KB per
// tile instead of 3.6 KB), so it does not depend on the motion-vector representation: one launch per batch.
//
// Work split: the unit of deblocking work is a SEGMENT (4 lines of one edge).  The 160 threads of a CTA take one
// segment each in four phases -- luma vertical (17 edge columns x 8 = 136 tasks), chroma vertical (2 planes x 9 x 8 = 144),
// luma horizontal (4 edge rows x 32 = 128), chroma horizontal (2 x 2 x 32 = 128) -- and a segment without an edge (zero record)
// costs a few instructions.  The fifth warp has vertical tasks only: its first thread draws the next tile from the queue while the
// other four run the horizontal pass.
// A chroma plane with the skip bit in its picture's control word (ilf_set_deblock_info found no intra unit: chroma is filtered
// for bS == 2 only, so the plane would come out unchanged) is not loaded, filtered or stored; it stays in the upload buffer.  When
// both are skipped the chroma records are not loaded either.
#include <algorithm>
#include <cstdlib>

#include "ilf_common.cuh"
#include "ilf_ring.cuh"

namespace ilf {
namespace {

constexpr int TW = RING_TILE_W, TH = DB_BAND_ROWS;  // luma tile; the band is shifted up by 4 rows
constexpr int CTW = TW / 2, CTH = TH / 2;           // chroma tile per plane; shifted up by 2 rows
constexpr int UW = TW / 4, UH = TH / 4;             // units per tile: 32 x 8, rows shifted up by 1
constexpr int BW = DB_BOX_W, BCW = DB_BOX_CW, BUW = DB_BOX_UNITS;   // box widths: the tile plus 8 samples (4 units) on each side
constexpr int MV16_UNITS = DB_BOX_MV16_WORDS / 2, MV32_UNITS = DB_BOX_MV32_WORDS / 4;   // motion boxes start at unit ux0 - 2 / ux0 - 1
// ILF_DB_STCS=1: results leave with st.global.cs (streaming, evict-first) stores.
#ifndef ILF_DB_STCS
#define ILF_DB_STCS 0
#endif
// ILF_DB_WIDE=1: 288 threads -- the luma and the chroma tasks of a phase run side by side (136 + 144 vertical, 128 + 128 horizontal)
// instead of one after the other.
#ifndef ILF_DB_WIDE
#define ILF_DB_WIDE 0
#endif
constexpr int NTHREADS = ILF_DB_WIDE ? 288 : 160;   // 136 / 144 vertical-edge tasks in one round; the horizontal passes use 128 of them
constexpr int VC0 = ILF_DB_WIDE ? 136 : 0, HC0 = ILF_DB_WIDE ? 128 : 0;   // first thread of the chroma tasks of the vertical / horizontal phase
// Ring depth and residency (measured, 17 4K pictures): 3 stages x 3 CTAs per SM 0.237 ms, 2 x 4 0.206 ms, 2 x 5 0.194 ms -- the kernel
// is bound by the latency of a tile's dependent phases, so more, smaller CTAs win over deeper prefetch.  With edge records instead of
// grid and motion boxes (15.4 KB stages, ra_4k stream decisions, B200): 2 x 5 0.1328 ms (66 registers), 2 x 6 0.1286 ms (59 registers,
// no spills), 3 x 5 0.1412 ms, 3 stages at a bound of 6 (4 fit by shared memory) 0.1414 ms.
#ifndef ILF_DB_STAGES
#define ILF_DB_STAGES 2
#endif
#ifndef ILF_DB_MIN_CTAS
#define ILF_DB_MIN_CTAS 6
#endif
constexpr int DB_STAGES = ILF_DB_STAGES;            // ring depth: the tile being filtered + DB_STAGES - 1 in flight (>= 2)
static_assert(DB_STAGES >= 2 && DB_STAGES <= 8, "a stage's next tile id is read one step after it was written only behind a barrier when there are two or more stages");

__constant__ uint8_t c_tc[66] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  1,  1,  1,  1,
                                 1,  1,  1,  1,  1,  2,  2,  2,  2,  3,  3,  3,  3,  4,  4,  4,  5,  5,  6,  6,  7,  8,
                                 9,  10, 11, 13, 14, 16, 18, 20, 22, 24, 26, 28, 30, 32, 34, 36, 38, 40, 42, 44, 46, 48};
__constant__ uint8_t c_beta[64] = {0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  6,  7,  8,  9,  10, 11,
                                   12, 13, 14, 15, 16, 17, 18, 20, 22, 24, 26, 28, 30, 32, 34, 36, 38, 40, 42, 44, 46, 48,
                                   50, 52, 54, 56, 58, 60, 62, 64, 66, 68, 70, 72, 74, 76, 78, 80, 82, 84, 86, 88};
__constant__ uint8_t c_chroma_scale[70] = {0,  1,  2,  3,  4,  5,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15, 16, 17,
                                           18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 29, 30, 31, 32, 33, 33,
                                           34, 34, 35, 35, 36, 36, 37, 37, 38, 39, 40, 41, 42, 43, 44, 45, 46, 47,
                                           48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61, 62, 63};

template <int MV> struct MvT { uint32_t dummy; };
template <> struct MvT<1> { uint2 v; };   // int16 x 4 per unit
template <> struct MvT<2> { int4 v; };    // int32 x 4 per unit
template <int MV> struct MvBox { static constexpr int UNITS = 1, OFF = 0; };
template <> struct MvBox<1> { static constexpr int UNITS = MV16_UNITS, OFF = 2; };
template <> struct MvBox<2> { static constexpr int UNITS = MV32_UNITS, OFF = 1; };

template <int MV> __device__ __forceinline__ void mv_get(const MvT<MV>& v, int m[4]);
template <> __device__ __forceinline__ void mv_get<0>(const MvT<0>&, int m[4]) { m[0] = m[1] = m[2] = m[3] = 0; }
template <> __device__ __forceinline__ void mv_get<1>(const MvT<1>& t, int m[4]) {
  m[0] = (int)(int16_t)(t.v.x & 0xFFFF); m[1] = (int)(int16_t)(t.v.x >> 16); m[2] = (int)(int16_t)(t.v.y & 0xFFFF); m[3] = (int)(int16_t)(t.v.y >> 16);
}
template <> __device__ __forceinline__ void mv_get<2>(const MvT<2>& t, int m[4]) { m[0] = t.v.x; m[1] = t.v.y; m[2] = t.v.z; m[3] = t.v.w; }

// A stage of the offset search = what the TMA unit delivers for a tile (dense boxes, each 128-byte aligned): sample column c of the
// tile is box column c + 8, unit column c is box column c + 4 (motion: c + 2 / c + 1).
template <int MV>
struct Stage {
  int16_t y[TH][BW];
  int16_t c[2][CTH][BCW];
  uint32_t info[UH][BUW];
  uint32_t info_c[UH][BUW];
  MvT<MV> mv[MV ? UH : 1][MvBox<MV>::UNITS];
};
static_assert(sizeof(int16_t[TH][BW]) % 128 == 0 && sizeof(int16_t[CTH][BCW]) % 128 == 0 && sizeof(uint32_t[UH][BUW]) % 128 == 0, "TMA destinations are 128-byte aligned");
template <int MV> __host__ __device__ constexpr int stage_stride() { return (int)((sizeof(Stage<MV>) + 127) & ~size_t(127)); }
template <int MV> __host__ __device__ constexpr int stage_tx_bytes(bool ctree) {
  return TH * BW * 2 + 2 * CTH * BCW * 2 + UH * BUW * 4 + (ctree ? UH * BUW * 4 : 0) + (MV == 1 ? UH * MV16_UNITS * 8 : (MV == 2 ? UH * MV32_UNITS * 16 : 0));
}

// The tile's window: unit columns -1 .. 32, sample columns -4 .. 131 (chroma -2 .. 65) are in the stage; what lies outside
// the picture arrives as zeros (no unit flags there, so nothing is filtered against it).
template <int MV>
struct Tile {
  Stage<MV>* st;
  bool ctree;
  __device__ __forceinline__ uint32_t info(int r, int c) const { return st->info[r][c + 4]; }
  __device__ __forceinline__ uint32_t cinfo(int r, int c) const { return ctree ? st->info_c[r][c + 4] : st->info[r][c + 4]; }
  __device__ __forceinline__ void mvs(int r, int c, int m[4]) const { mv_get<MV>(st->mv[MV ? r : 0][MV ? c + MvBox<MV>::OFF : 0], m); }
  __device__ __forceinline__ int16_t* y(int r, int c) const { return &st->y[r][c + 8]; }
  __device__ __forceinline__ int16_t* ch(int pl, int r, int c) const { return &st->c[pl][r][c + 8]; }
};

// The same accessors over the slot's side information in device memory (the record pass): unit (r, c) of the held rows; what
// lies outside them reads as zeros, as outside the picture in a TMA box.
struct Grid {
  const uint32_t* units;
  const uint32_t* units_c;  // chroma-tree layer or nullptr
  const int16_t* mv16;      // at most one of the two; neither: every unit intra, no vector is read
  const int32_t* mv32;
  int units_w, units_h, pitch;
  __device__ __forceinline__ bool in(int r, int c) const { return r >= 0 && r < units_h && c >= 0 && c < units_w; }
  __device__ __forceinline__ uint32_t info(int r, int c) const { return in(r, c) ? __ldg(units + (size_t)r * pitch + c) : 0u; }
  __device__ __forceinline__ uint32_t cinfo(int r, int c) const { return in(r, c) ? __ldg((units_c ? units_c : units) + (size_t)r * pitch + c) : 0u; }
  __device__ __forceinline__ void mvs(int r, int c, int m[4]) const {
    MvT<2> v = {make_int4(0, 0, 0, 0)};
    if (in(r, c) && mv32) v.v = __ldg(reinterpret_cast<const int4*>(mv32) + (size_t)r * pitch + c);
    if (in(r, c) && mv16) {
      const uint2 w = __ldg(reinterpret_cast<const uint2*>(mv16) + (size_t)r * pitch + c);
      v.v = make_int4((int16_t)(w.x & 0xFFFF), (int16_t)(w.x >> 16), (int16_t)(w.y & 0xFFFF), (int16_t)(w.y >> 16));
    }
    mv_get<2>(v, m);
  }
};

// bS of one 4-sample segment (xGetBoundaryStrengthSingle, LoopFilter.cpp:419-541).  q, p index the view (Tile or Grid).
template <class View>
__device__ __forceinline__ int boundary_strength(const View& t, uint32_t iq, uint32_t ip, int qr, int qc, int pr, int pc, uint32_t tu_bit, int thr) {
  if ((iq | ip) & ILF_BI_INTRA) return 2;
  if ((iq & tu_bit) && ((iq | ip) & ILF_BI_CBF)) return 1;
  const int rq0 = (iq >> 16) & 0xFF, rq1 = iq >> 24, rp0 = (ip >> 16) & 0xFF, rp1 = ip >> 24;
  int mq[4], mp[4];
  t.mvs(qr, qc, mq);
  t.mvs(pr, pc, mp);
  const bool d00 = abs(mq[0] - mp[0]) >= thr || abs(mq[1] - mp[1]) >= thr;
  if ((iq | ip) & ILF_BI_BSLICE) {
    if ((rp0 == rq0 && rp1 == rq1) || (rp0 == rq1 && rp1 == rq0)) {
      const bool d11 = abs(mq[2] - mp[2]) >= thr || abs(mq[3] - mp[3]) >= thr;
      const bool d10 = abs(mq[2] - mp[0]) >= thr || abs(mq[3] - mp[1]) >= thr;
      const bool d01 = abs(mq[0] - mp[2]) >= thr || abs(mq[1] - mp[3]) >= thr;
      if (rp0 != rp1) return (rp0 == rq0) ? (d00 || d11) : (d10 || d01);
      return (d00 || d11) && (d10 || d01);
    }
    return 1;
  }
  if (rp0 != rq0) return 1;
  return d00;
}

// Luma filter of one line across an edge (xPelFilterLuma, LoopFilter.cpp:856-916).  v[0..7] = p3 p2 p1 p0 | q0 q1 q2 q3.
__device__ __forceinline__ void filter_luma_line(int v[8], int tc, bool sw, bool no_p, bool no_q, int thr_cut, bool second_p, bool second_q, int max_val) {
  const int m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3], m4 = v[4], m5 = v[5], m6 = v[6], m7 = v[7];
  if (sw) {
    const int t2 = 2 * tc;
    v[3] = clip3i(m3 - t2, m3 + t2, (m1 + 2 * m2 + 2 * m3 + 2 * m4 + m5 + 4) >> 3);
    v[4] = clip3i(m4 - t2, m4 + t2, (m2 + 2 * m3 + 2 * m4 + 2 * m5 + m6 + 4) >> 3);
    v[2] = clip3i(m2 - t2, m2 + t2, (m1 + m2 + m3 + m4 + 2) >> 2);
    v[5] = clip3i(m5 - t2, m5 + t2, (m3 + m4 + m5 + m6 + 2) >> 2);
    v[1] = clip3i(m1 - t2, m1 + t2, (2 * m0 + 3 * m1 + m2 + m3 + m4 + 4) >> 3);
    v[6] = clip3i(m6 - t2, m6 + t2, (m3 + m4 + m5 + 3 * m6 + 2 * m7 + 4) >> 3);
  } else {
    int delta = (9 * (m4 - m3) - 3 * (m5 - m2) + 8) >> 4;
    if (abs(delta) < thr_cut) {
      delta = clip3i(-tc, tc, delta);
      v[3] = clip3i(0, max_val, m3 + delta);
      v[4] = clip3i(0, max_val, m4 - delta);
      const int tc2 = tc >> 1;
      if (second_p) v[2] = clip3i(0, max_val, m2 + clip3i(-tc2, tc2, (((m1 + m3 + 1) >> 1) - m2 + delta) >> 1));
      if (second_q) v[5] = clip3i(0, max_val, m5 + clip3i(-tc2, tc2, (((m6 + m4 + 1) >> 1) - m5 - delta) >> 1));
    }
  }
  if (no_p) { v[3] = m3; v[2] = m2; v[1] = m1; }
  if (no_q) { v[4] = m4; v[5] = m5; v[6] = m6; }
}

struct EdgeParams {
  int bs;        // 0 = leave the segment alone
  int tc, beta;
  bool no_p, no_q;
};

// Offset-independent part of a luma segment (xEdgeFilterLuma, LoopFilter.cpp:543-634, up to the tables): 0 = not filtered, else
// bS | no_p << 2 | no_q << 3 | (QP & 0xFF) << 8.  (qr, qc) / (pr, pc) = unit row and column of the Q / P unit in the view.
template <class View>
__device__ __forceinline__ uint32_t luma_edge_record(const View& t, int thr, int qr, int qc, int pr, int pc, bool vertical) {
  const uint32_t iq = t.info(qr, qc), ip = t.info(pr, pc);
  if (!(iq & (vertical ? ILF_BI_EDGE_V : ILF_BI_EDGE_H))) return 0;
  const int bs = boundary_strength(t, iq, ip, qr, qc, pr, pc, vertical ? ILF_BI_TU_V : ILF_BI_TU_H, thr);
  if (!bs) return 0;
  const int qp = ((int)(int8_t)(ip >> 8) + (int)(int8_t)(iq >> 8) + 1) >> 1;
  return (uint32_t)bs | ((ip & ILF_BI_NOFILT) ? 4u : 0u) | ((iq & ILF_BI_NOFILT) ? 8u : 0u) | ((uint32_t)(qp & 0xFF) << 8);
}

// Offset-independent part of a chroma segment (xEdgeFilterChroma, LoopFilter.cpp:684-838, up to the table): 0 = not filtered, else
// 1 | no_p << 1 | no_q << 2 | (chroma QP after the mapping) << 16.
__device__ __forceinline__ uint32_t chroma_edge_record(uint32_t iq, uint32_t ip, const ilf_deblock_params& prm, const uint8_t* chroma_scale, bool vertical, int comp) {
  if (!(iq & (vertical ? ILF_BI_EDGE_V : ILF_BI_EDGE_H))) return 0;
  if (!((iq | ip) & ILF_BI_INTRA)) return 0;  // chroma is filtered for bS == 2 only (:769)
  int qp = (((int)(int8_t)(ip >> 8) + (int)(int8_t)(iq >> 8) + 1) >> 1) + (comp == 0 ? prm.cb_qp_offset : prm.cr_qp_offset);
  if (qp >= 70) qp -= 6;
  else if (qp >= 0) qp = chroma_scale[qp];
  return 1u | ((ip & ILF_BI_NOFILT) ? 2u : 0u) | ((iq & ILF_BI_NOFILT) ? 4u : 0u) | ((uint32_t)qp << 16);
}

// ---------------------------------------------------------------------------------------------------------------------------
// Record pass (ilf_set_deblock_info).  A segment's 16-bit record, 0 = nothing to filter:
//   luma    1 | no_p << 1 | no_q << 2 | tc index << 3 | beta index << 10   (indices into c_tc / c_beta, slice offsets applied)
//   chroma  1 | no_p << 1 | no_q << 2 | tc index << 3                      (per plane: QP offset and mapping applied)
// deblock_kernel multiplies the table values by the bit-depth scale.
__device__ __forceinline__ uint32_t luma_record(uint32_t r, const ilf_slice_params& sl) {
  if (!r) return 0;
  const int bs = r & 3, qp = (int)(int8_t)(r >> 8);
  const int tci = clip3i(0, 65, qp + 2 * (bs - 1) + 2 * sl.tc_offset_div2), bi = clip3i(0, 63, qp + 2 * sl.beta_offset_div2);
  return 1u | ((r & 4) ? 2u : 0u) | ((r & 8) ? 4u : 0u) | (uint32_t)tci << 3 | (uint32_t)bi << 10;
}
__device__ __forceinline__ uint32_t chroma_record(uint32_t r, const ilf_slice_params& sl) {
  if (!r) return 0;
  return 1u | (r & 6u) | (uint32_t)clip3i(0, 65, ((int)r >> 16) + 2 + 2 * sl.tc_offset_div2) << 3;
}

// One thread per record; blockIdx.y = DB_REC_* kind.  Coordinates: unit rows / columns of the held rows, slices looked up at the
// full-picture position of the segment's first Q sample.
__global__ void __launch_bounds__(256) deblock_records_kernel(Geom g, Grid grid, const ilf_deblock_params* __restrict__ params, const uint8_t* __restrict__ ctu_slice,
                                                              const __grid_constant__ DbRecLayout L, unsigned char* __restrict__ rec) {
  __shared__ ilf_deblock_params prm;
  __shared__ uint8_t chroma_scale[70 + 2];
  for (int i = threadIdx.x; i < (int)(sizeof(ilf_deblock_params) / 4); i += blockDim.x) reinterpret_cast<uint32_t*>(&prm)[i] = __ldg(reinterpret_cast<const uint32_t*>(params) + i);
  if (threadIdx.x < 70) chroma_scale[threadIdx.x] = c_chroma_scale[threadIdx.x];
  __syncthreads();
  const int k = blockIdx.y, cols = L.cols[k], n = cols * L.rows[k];
  auto slice = [&](int xg, int yg) -> const ilf_slice_params& {
    return prm.slices[ctu_slice ? (int)__ldg(ctu_slice + (size_t)((yg + g.row0) >> g.ctu_log2) * g.ctus_w + (xg >> g.ctu_log2)) : 0];
  };
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int r = i / cols, c = i - r * cols;
    unsigned char* out = rec + L.off[k] + ((size_t)r * L.pitch[k] + c) * L.elem[k];
    if (k == DB_REC_LV) {        // edge x = 8 c, unit row r
      const uint32_t e = luma_edge_record(grid, prm.mv_threshold, r, 2 * c, r, 2 * c - 1, true);
      *reinterpret_cast<uint16_t*>(out) = (uint16_t)(e ? luma_record(e, slice(8 * c, 4 * r)) : 0);
    } else if (k == DB_REC_LH) { // edge y = 8 r, unit column c
      const uint32_t e = luma_edge_record(grid, prm.mv_threshold, 2 * r, c, 2 * r - 1, c, false);
      *reinterpret_cast<uint16_t*>(out) = (uint16_t)(e ? luma_record(e, slice(4 * c, 8 * r)) : 0);
    } else {                     // chroma edge cx = 8 c (luma 16 c), unit row r / cy = 8 r (luma 16 r), unit column c
      const bool v = k == DB_REC_CV;
      const int qr = v ? r : 4 * r, qc = v ? 4 * c : c, pr = v ? r : 4 * r - 1, pc = v ? 4 * c - 1 : c;
      const uint32_t iq = grid.cinfo(qr, qc), ip = grid.cinfo(pr, pc);
      uint32_t w = 0;
      for (int pl = 0; pl < 2; pl++) {
        const uint32_t e = chroma_edge_record(iq, ip, prm, chroma_scale, v, pl);
        if (e) w |= chroma_record(e, slice(v ? 16 * c : 4 * c, v ? 4 * r : 16 * r)) << (16 * pl);
      }
      *reinterpret_cast<uint32_t*>(out) = w;
    }
  }
}

// The tc / beta tables and the per-picture destination, copied to shared memory once per CTA: the segments index the tables with
// per-thread values (constant memory would serialise).
struct DbShared {
  int tile[8];               // tile in (or on its way into) every stage of the ring: tx | ty << 8 | z << 20, -1 = the queue is empty
  int cur_slot;              // grid layer whose destination is in dst / ctl
  int next;                  // tile drawn for the stage that is being emptied
  int16_t* dst[3];           // destination planes and control word of grid layer cur_slot
  unsigned ctl;
  uint8_t tc[66 + 2], beta[64];
};

// A luma record -> the segment's parameters (LoopFilter.cpp:626-634).
__device__ __forceinline__ EdgeParams luma_edge(uint32_t rec, const DbShared& sh, int scale) {
  EdgeParams ep;
  ep.bs = 1;
  ep.tc = sh.tc[(rec >> 3) & 127] * scale;
  ep.beta = sh.beta[rec >> 10] * scale;
  ep.no_p = (rec & 2) != 0;
  ep.no_q = (rec & 4) != 0;
  return ep;
}

// Decisions of a segment from its lines 0 and 3 (LoopFilter.cpp:640-671) and filtering of its four lines.
// L[i][0..7] = line i of the segment, p3 p2 p1 p0 | q0 q1 q2 q3.  Returns false when nothing was changed.
__device__ __forceinline__ bool filter_luma_segment(int (&L)[4][8], const EdgeParams& ep, int max_val) {
  const int dp0 = abs(L[0][1] - 2 * L[0][2] + L[0][3]), dq0 = abs(L[0][4] - 2 * L[0][5] + L[0][6]);
  const int dp3 = abs(L[3][1] - 2 * L[3][2] + L[3][3]), dq3 = abs(L[3][4] - 2 * L[3][5] + L[3][6]);
  const int d0 = dp0 + dq0, d3 = dp3 + dq3;
  if (d0 + d3 >= ep.beta) return false;
  const int side_thr = (ep.beta + (ep.beta >> 1)) >> 3;
  const bool second_p = (dp0 + dp3) < side_thr, second_q = (dq0 + dq3) < side_thr;
  // xUseStrongFiltering on lines 0 and 3 with d = 2 * d0 / 2 * d3 (:670-671, :960-970)
  const int tc52 = (ep.tc * 5 + 1) >> 1;
  const bool s0 = (abs(L[0][0] - L[0][3]) + abs(L[0][7] - L[0][4]) < (ep.beta >> 3)) && (2 * d0 < (ep.beta >> 2)) && (abs(L[0][3] - L[0][4]) < tc52);
  const bool s3 = (abs(L[3][0] - L[3][3]) + abs(L[3][7] - L[3][4]) < (ep.beta >> 3)) && (2 * d3 < (ep.beta >> 2)) && (abs(L[3][3] - L[3][4]) < tc52);
  const bool sw = s0 && s3;
#pragma unroll
  for (int i = 0; i < 4; i++) filter_luma_line(L[i], ep.tc, sw, ep.no_p, ep.no_q, ep.tc * 10, second_p, second_q, max_val);
  return true;
}

__device__ __forceinline__ void unpack2(uint32_t w, int& a, int& b) { a = (int)(int16_t)(w & 0xFFFF); b = (int)(int16_t)(w >> 16); }
__device__ __forceinline__ uint32_t pack2(int a, int b) { return (uint32_t)(uint16_t)a | ((uint32_t)b << 16); }

// One stage of deblock_kernel = what the TMA unit delivers for a tile (dense boxes, each 128-byte aligned): sample column c of the
// tile is box column c + 8; the record boxes start at the tile's first edge column and first segment row (ilf_common.cuh).
struct DbStage {
  int16_t y[TH][BW];
  int16_t c[2][CTH][BCW];
  uint16_t rec_lv[DB_REC_LV_H][DB_REC_LV_W];   // [segment row sg][edge e]: x0 + 8 e, rows y0 + 4 sg ..
  uint16_t rec_lh[DB_REC_LH_H][DB_REC_LH_W];   // [edge row h][unit column u]: y0 + 4 + 8 h, columns x0 + 4 u ..
  uint32_t rec_cv[DB_REC_CV_H][DB_REC_CV_W];   // [segment row sg][edge k]: cx0 + 8 k, chroma rows cy0 + 2 sg .. (Cb | Cr << 16)
  uint32_t rec_ch[DB_REC_CH_H][DB_REC_CH_W];   // [edge row h][unit column u]: cy0 + 2 + 8 h, chroma columns cx0 + 2 u ..
};
static_assert(sizeof(int16_t[TH][BW]) % 128 == 0 && sizeof(int16_t[CTH][BCW]) % 128 == 0 && sizeof(uint16_t[DB_REC_LV_H][DB_REC_LV_W]) % 128 == 0 &&
              sizeof(uint16_t[DB_REC_LH_H][DB_REC_LH_W]) % 128 == 0 && sizeof(uint32_t[DB_REC_CV_H][DB_REC_CV_W]) % 128 == 0, "TMA destinations are 128-byte aligned");
static_assert(DB_REC_LV_W >= TW / 8 + 1 && DB_REC_CV_W >= CTW / 8 + 1, "a vertical record box holds the tile's edges and the next tile's first");
constexpr int DB_STRIDE = (int)((sizeof(DbStage) + 127) & ~size_t(127));
constexpr int DB_REC_LUMA_BYTES = (int)(sizeof(DbStage::rec_lv) + sizeof(DbStage::rec_lh)), DB_REC_CHROMA_BYTES = (int)(sizeof(DbStage::rec_cv) + sizeof(DbStage::rec_ch));

__global__ void __launch_bounds__(NTHREADS, ILF_DB_MIN_CTAS) deblock_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc, int num_slots, int* __restrict__ work) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int S = DB_STAGES;
  pdl_launch_dependents();
  const int tid = threadIdx.x;
  const int rows = g.rows, crow = g.rows >> 1, cw = g.width >> 1;
  const int ntx = (g.width + TW - 1) / TW, bands = (g.rows + 4 + TH - 1) / TH;
  const int total = ntx * bands * num_slots;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S * DB_STRIDE);
  DbShared& sh = *reinterpret_cast<DbShared*>(smem + S * DB_STRIDE + 8 * S);
  // tile id -> (grid layer, band, tile of the band): raster order inside a picture, pictures one after the other
  auto pack_id = [&](int id) { if (id >= total) return -1; const int tx = id % ntx, r = id / ntx; return tx | (r % bands) << 8 | (r / bands) << 20; };
  auto decode = [&](int id, int& z, int& ty, int& tx) { tx = id & 255; ty = (id >> 8) & 4095; z = id >> 20; };
  // The boxes of a tile are issued by the first lanes of the CTA's warps, one part each, so that their descriptor fetches
  // overlap: part 0 arms the barrier and loads luma, 1 both chroma planes, 2 the luma records, 3 the chroma records.  A skipped
  // chroma plane (a picture without an intra unit: no chroma edge is filtered) is neither loaded nor stored, and with both planes
  // skipped the chroma records stay behind too.  The tile may belong to another picture than sh.cur_slot, so its control word is
  // read from bc.
  auto issue_part = [&](int id, int si, int part) {  // tile id into stage si
    int z, ty, tx;
    decode(id, z, ty, tx);
    const SlotDev& sd = slots[first_slot + bc.slot[z]];
    const unsigned c = bc.v[z];
    const bool chroma = !(ctl_skip(c, 1) && ctl_skip(c, 2));
    DbStage* st = reinterpret_cast<DbStage*>(smem + si * DB_STRIDE);
    uint64_t* bar = &full[si];
    if (part == 0) {
      const int skipped = (int)ctl_skip(c, 1) + (int)ctl_skip(c, 2);
      ring::mbar_expect_tx(bar, (uint32_t)(TH * BW * 2 + (2 - skipped) * (CTH * BCW * 2) + DB_REC_LUMA_BYTES + (chroma ? DB_REC_CHROMA_BYTES : 0)));
      ring::tma_load_3d(&st->y[0][0], &sd.tm_db[0], bar, tx * TW - 8, ty * TH - 4, ctl_src(c, 0));
    } else if (part == 1) {
      if (!ctl_skip(c, 1)) ring::tma_load_3d(&st->c[0][0][0], &sd.tm_db[1], bar, tx * CTW - 8, ty * CTH - 2, ctl_src(c, 0));
      if (!ctl_skip(c, 2)) ring::tma_load_3d(&st->c[1][0][0], &sd.tm_db[2], bar, tx * CTW - 8, ty * CTH - 2, ctl_src(c, 0));
    } else if (part == 2) {
      ring::tma_load_3d(&st->rec_lv[0][0], &sd.tm_rec[DB_REC_LV], bar, tx * (TW / 8), ty * UH - 1, 0);
      ring::tma_load_3d(&st->rec_lh[0][0], &sd.tm_rec[DB_REC_LH], bar, tx * UW, ty * (TH / 8), 0);
    } else if (chroma) {
      ring::tma_load_3d(&st->rec_cv[0][0], &sd.tm_rec[DB_REC_CV], bar, tx * (CTW / 8), ty * UH - 1, 0);
      ring::tma_load_3d(&st->rec_ch[0][0], &sd.tm_rec[DB_REC_CH], bar, tx * UW, ty * (TH / 16), 0);
    }
  };
  if (tid == 0) {
    for (int i = 0; i < S; i++) ring::mbar_init(&full[i], 1);
    ring::mbar_init_fence();
    sh.cur_slot = -1;
  }
  if (tid < 66) sh.tc[tid] = c_tc[tid];
  if (tid < 64) sh.beta[tid] = c_beta[tid];
  pdl_wait();  // the previous chain's last stage has finished with the buffers this stage reads and writes -- and has reset the work counter
  // Work queue: tiles are drawn from one counter in raster order, so the CTAs resident at any moment work on a compact window of
  // the picture whatever their relative progress; a CTA keeps S - 1 tiles in flight ahead of the one it filters.
  if (tid == 0)
    for (int i = 0; i < S; i++) sh.tile[i] = pack_id(atomicAdd(&work[0], 1));
  __syncthreads();
  if ((tid & 31) == 0)
    for (int i = 0; i < S; i++) if (sh.tile[i] >= 0 && tid < 128) issue_part(sh.tile[i], i, tid >> 5);

  const int max_y = (1 << g.bd_luma) - 1, max_c = (1 << g.bd_chroma) - 1;
  const int scale_y = 1 << (g.bd_luma - 8), scale_c = 1 << (g.bd_chroma - 8);
  const bool filt = !(g.debug & 1);
  int si = 0;
  uint32_t phases = 0;   // bit s: parity of stage s's next completion
  for (;;) {
    const int id = sh.tile[si];
    if (id < 0) break;
    int z, ty, tx;
    decode(id, z, ty, tx);
    if (sh.cur_slot != z) {   // CTA-uniform: the picture's destination -> shared memory (once per picture a CTA meets)
      __syncthreads();
      if (tid == 0) {
        const SlotDev& sd = slots[first_slot + bc.slot[z]];
        const unsigned c = bc.v[z];
        const int db = ctl_dst(c, 0);  // deblocking starts from the uploaded picture: all planes in one buffer (skipped planes are not written)
        sh.ctl = c; sh.dst[0] = sd.buf[db][0]; sh.dst[1] = sd.buf[db][1]; sh.dst[2] = sd.buf[db][2];
        sh.cur_slot = z;
      }
      __syncthreads();
    }
    const int y0 = ty * TH - 4, cy0 = ty * CTH - 2;
    int16_t* __restrict__ dst_y = sh.dst[0];
    int16_t* __restrict__ dst_cb = sh.dst[1];
    int16_t* __restrict__ dst_cr = sh.dst[2];
    DbStage* const st = reinterpret_cast<DbStage*>(smem + si * DB_STRIDE);
    ring::mbar_wait(&full[si], (phases >> si) & 1u);
    phases ^= 1u << si;
    const int x0 = tx * TW, cx0 = tx * CTW;

    // ---- vertical edges, luma: task = 4 lines x 8 samples.  17 edge columns x 8 segment rows (tasks 128 .. 135: edge 16) ----
    if (filt) {
      if (tid < 17 * 8) {
        const int task = tid;
        const int e = task < 128 ? (task & 15) : 16, sg = task < 128 ? (task >> 4) : task - 128;
        const uint32_t rec = st->rec_lv[sg][e];
        if (rec) {
          const EdgeParams ep = luma_edge(rec, sh, scale_y);
          int16_t* pp = &st->y[4 * sg][8 * e + 4];
          int16_t* pq = &st->y[4 * sg][8 * e + 8];
          int L[4][8];
#pragma unroll
          for (int i = 0; i < 4; i++) {
            const uint2 a = *reinterpret_cast<const uint2*>(pp + i * BW), b = *reinterpret_cast<const uint2*>(pq + i * BW);
            unpack2(a.x, L[i][0], L[i][1]); unpack2(a.y, L[i][2], L[i][3]); unpack2(b.x, L[i][4], L[i][5]); unpack2(b.y, L[i][6], L[i][7]);
          }
          if (filter_luma_segment(L, ep, max_y)) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
              *reinterpret_cast<uint2*>(pp + i * BW) = make_uint2(pack2(L[i][0], L[i][1]), pack2(L[i][2], L[i][3]));
              *reinterpret_cast<uint2*>(pq + i * BW) = make_uint2(pack2(L[i][4], L[i][5]), pack2(L[i][6], L[i][7]));
            }
          }
        }
      }
      // ---- vertical edges, chroma: task = one unit = 2 lines x 4 samples.  2 planes x 9 edge columns x 8 unit rows (tasks 128 .. 143: edge 8) ----
      const int task = tid - VC0;
      const int pl = task < 128 ? (task >> 6) : ((task - 128) >> 3);
      if (tid >= VC0 && task < 2 * 9 * 8 && !ctl_skip(sh.ctl, 1 + pl)) {
        const int k = task < 128 ? ((task >> 3) & 7) : 8, sg = task & 7;
        const uint32_t rec = (st->rec_cv[sg][k] >> (16 * pl)) & 0xFFFFu;
        if (rec) {
          const int tc = sh.tc[rec >> 3] * scale_c;
          const bool no_p = rec & 2, no_q = rec & 4;
          int16_t* pp = &st->c[pl][2 * sg][8 * k + 6];
          int16_t* pq = &st->c[pl][2 * sg][8 * k + 8];
#pragma unroll
          for (int i = 0; i < 2; i++) {
            const int m2 = pp[i * BCW], m3 = pp[i * BCW + 1], m4 = pq[i * BCW], m5 = pq[i * BCW + 1];
            const int delta = clip3i(-tc, tc, (((m4 - m3) << 2) + m2 - m5 + 4) >> 3);
            if (!no_p) pp[i * BCW + 1] = (int16_t)clip3i(0, max_c, m3 + delta);
            if (!no_q) pq[i * BCW] = (int16_t)clip3i(0, max_c, m4 - delta);
          }
        }
      }
    }
    __syncthreads();
    // the tile that will take this stage is drawn by the first thread of the last warp, which has no horizontal task: the
    // atomic's latency and the division of the id stay off the path of the warps that filter
    if (tid == NTHREADS - 32) sh.next = pack_id(atomicAdd(&work[0], 1));

    // ---- horizontal edges, luma: task = 4 columns x 8 rows, filtered and stored.  4 edge rows x 32 unit columns
    //      (a warp = one edge row: 256 contiguous bytes per stored row) ----
    if (tid < 128) {
      const int u = tid & 31, h = tid >> 5;
      const int16_t* sp = &st->y[8 * h][4 * u + 8];
      uint2 raw[8];
#pragma unroll
      for (int i = 0; i < 8; i++) raw[i] = *reinterpret_cast<const uint2*>(sp + i * BW);
      const uint32_t rec = st->rec_lh[h][u];
      if (filt && rec) {
        const EdgeParams ep = luma_edge(rec, sh, scale_y);
        int L[4][8];
#pragma unroll
        for (int i = 0; i < 8; i++) { unpack2(raw[i].x, L[0][i], L[1][i]); unpack2(raw[i].y, L[2][i], L[3][i]); }
        if (filter_luma_segment(L, ep, max_y)) {
#pragma unroll
          for (int i = 1; i < 7; i++) raw[i] = make_uint2(pack2(L[0][i], L[1][i]), pack2(L[2][i], L[3][i]));
        }
      }
      const int x = x0 + 4 * u;
      if (x < g.width) {
        int16_t* op = dst_y + (size_t)(y0 + 8 * h) * g.pitch_y + x;
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int y = y0 + 8 * h + i;
          if (y >= 0 && y < rows) {
#if ILF_DB_STCS
            __stcs(reinterpret_cast<uint2*>(op + (size_t)i * g.pitch_y), raw[i]);
#else
            *reinterpret_cast<uint2*>(op + (size_t)i * g.pitch_y) = raw[i];
#endif
          }
        }
      }
    }
    // ---- horizontal edges, chroma: task = 2 columns x 8 rows (the edge lies between rows 1 and 2), filtered and stored.
    //      2 planes x 2 row groups x 32 unit columns ----
    if (tid >= HC0 && tid < HC0 + 128 && !ctl_skip(sh.ctl, 1 + ((tid - HC0) >> 6))) {
      const int ht = tid - HC0;
      const int pl = ht >> 6, h = (ht >> 5) & 1, u = ht & 31;
      const int16_t* sp = &st->c[pl][8 * h][2 * u + 8];
      uint32_t raw[8];
#pragma unroll
      for (int i = 0; i < 8; i++) raw[i] = *reinterpret_cast<const uint32_t*>(sp + i * BCW);
      const uint32_t rec = (st->rec_ch[h][u] >> (16 * pl)) & 0xFFFFu;
      if (filt && rec) {
        const int tc = sh.tc[rec >> 3] * scale_c;
        int a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; i++) unpack2(raw[i], a[i], b[i]);
        const int da = clip3i(-tc, tc, (((a[2] - a[1]) << 2) + a[0] - a[3] + 4) >> 3);
        const int db = clip3i(-tc, tc, (((b[2] - b[1]) << 2) + b[0] - b[3] + 4) >> 3);
        if (!(rec & 2)) raw[1] = pack2(clip3i(0, max_c, a[1] + da), clip3i(0, max_c, b[1] + db));
        if (!(rec & 4)) raw[2] = pack2(clip3i(0, max_c, a[2] - da), clip3i(0, max_c, b[2] - db));
      }
      const int x = cx0 + 2 * u;
      if (x < cw) {
        int16_t* op = (pl ? dst_cr : dst_cb) + (size_t)(cy0 + 8 * h) * g.pitch_c + x;
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int y = cy0 + 8 * h + i;
          if (y >= 0 && y < crow) {
#if ILF_DB_STCS
            __stcs(reinterpret_cast<uint32_t*>(op + (size_t)i * g.pitch_c), raw[i]);
#else
            *reinterpret_cast<uint32_t*>(op + (size_t)i * g.pitch_c) = raw[i];
#endif
          }
        }
      }
    }
    // every thread is done with the stage: it is refilled with the next tile of the queue
    __syncthreads();
    {
      const int nid = sh.next;
      if ((tid & 31) == 0 && tid < 128 && nid >= 0) issue_part(nid, si, tid >> 5);   // (four lanes of ONE warp would issue the parts one after the other: 0.1925 against 0.189 ms)
      if (tid == 0) sh.tile[si] = nid;   // read S steps from now, behind more barriers
    }
    if (++si == S) si = 0;
  }
  // the last CTA to leave resets the queue for the next launch on this stream (every CTA has drawn its last id by now)
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(&work[1], 1) == (int)gridDim.x - 1) { work[0] = 0; work[1] = 0; __threadfence(); }
  }
}

}  // namespace

// work: two ints in device memory, zero before the first launch and owned by the launching stream (the kernel leaves them zero).
void launch_deblock(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, int* work, cudaStream_t st) {
  static const int pad = env_int("ILF_DB_SMEM_PAD");
  const int smem = DB_STAGES * DB_STRIDE + DB_STAGES * 8 + (int)sizeof(DbShared) + pad;
  static bool attr_set[64] = {};
  once_per_device(attr_set, [&] { cudaFuncSetAttribute(deblock_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
  const int bands = (g.rows + 4 + TH - 1) / TH, ntx = (g.width + TW - 1) / TW;
  const long long total = (long long)ntx * bands * num_slots;
  // CTAs drawing tiles from the queue: the resident ones plus a fifth.  Exactly the resident number starves the kernel when
  // another lane's CTAs hold slots (stream chain 0.290 ms); every CTA beyond those that ever get a slot while the queue is
  // non-empty only runs its prologue at the end of the launch (twice the resident number: 0.275 ms; 800 - 1000 CTAs: 0.271 ms).
  static const int ctas = env_int("ILF_DB_CTAS", 148 * (ILF_DB_MIN_CTAS + 1));
  dim3 grid((unsigned)std::min<long long>(total, ctas));
  launch_pdl(deblock_kernel, grid, dim3(NTHREADS), smem, st, g, slots, first_slot, ctl, num_slots, work);
}

void launch_deblock_records(const Geom& g, const ilf_deblock_params* params, const uint32_t* info, const uint32_t* info_c, const int16_t* mv16,
                            const int32_t* mv32, const uint8_t* ctu_slice, void* rec, cudaStream_t st) {
  const DbRecLayout L = db_rec_layout(g);
  const Grid grid = {info, info_c, mv16, mv32, g.units_w, g.units_h, g.units_pitch};
  int most = 0;
  for (int k = 0; k < DB_REC_KINDS; k++) most = std::max(most, L.cols[k] * L.rows[k]);
  const dim3 blocks((unsigned)std::min(std::max(1, (most + 255) / 256), 148 * 8), DB_REC_KINDS);
  deblock_records_kernel<<<blocks, 256, 0, st>>>(g, grid, params, ctu_slice, L, static_cast<unsigned char*>(rec));
}

// ---------------------------------------------------------------------------------------------------------------------------
// Deblocking offset search (ilf_deblock_search; EncGOP::applyDeblockingFilterParameterSelection).  The same tiles and device
// functions as deblock_kernel, but a tile is deblocked K times, once per (beta, tc) offset candidate, and nothing is
// stored: the horizontal-pass tasks compare their filtered block with the original and only sums of squared differences leave.
//   - the slot's edge records have the slice offsets applied, so the stage carries the unit grid and the motion vectors instead
//     (one launch per motion-vector representation), and per tile what does not depend on the offsets (edge flag, bS, QP,
//     no-filter sides, chroma QP) is derived once into a compact record per segment; a thread owns the same four segments (one per phase) for every candidate, so the records stay
//     in its registers, and so does the horizontal-pass task's block of the original;
//   - per candidate: the staged samples are copied into a work buffer (two buffers alternate, so the copy of candidate k + 1 needs
//     no barrier behind the horizontal pass of k), vertical edges, a barrier, horizontal edges + distortion;
//   - a tile without any filtered segment has the same distortion for every candidate: it is measured once (`common`);
//   - sums: a thread's block fits uint32 (32 x 4095^2 < 2^32), a warp's sum does not: 64-bit warp reduction, then per-warp rows
//     [candidate][plane] in shared memory (one writer each, no atomics), flushed to global memory with one 64-bit atomicAdd per
//     entry when the CTA moves on to another slot and at exit.
// The CTAs walk the tiles of a launch statically (tile blockIdx.x + i * gridDim.x): there is no work counter to share with
// deblocking launches on other streams.  A tile's K passes hide the fetch of the next tile, which is issued once the last
// candidate's copy is done.
namespace {

constexpr int SEARCH_MAX = ILF_DEBLOCK_SEARCH_MAX;
constexpr int SEARCH_THREADS = 160;   // the task split of deblock_kernel: 136 / 144 vertical tasks, 128 + 128 horizontal tasks on warps 0..3
constexpr int SEARCH_WARPS_H = 4;     // warps with horizontal tasks (luma: all four; Cb: warps 0, 1; Cr: warps 2, 3)
constexpr int SEARCH_MIN_CTAS = 4;    // 95 registers, no spills; about 55 KB of shared memory per CTA also fits four (123 registers, 3 CTAs, unbounded)

struct SearchCands {
  ilf_deblock_candidate c[SEARCH_MAX];
  int n;
  int shift_luma, shift_chroma;
};

// The sample part of a stage (its first bytes: luma, then both chroma planes, same layout), copied once per candidate.
struct SearchWork {
  int16_t y[TH][BW];
  int16_t c[2][CTH][BCW];
};
static_assert(sizeof(SearchWork) % 128 == 0 && sizeof(SearchWork) % 16 == 0, "work buffers are copied with 16-byte moves and stay 128-byte aligned");

struct SearchShared {
  unsigned long long acc[SEARCH_WARPS_H][SEARCH_MAX][3];   // per warp: [candidate][Y, Cb, Cr]
  unsigned long long common[SEARCH_WARPS_H][3];            // tiles without a filtered segment: the same for every candidate
  uint64_t full;                                           // the stage's barrier
  ilf_deblock_params prm;                                  // of the slot being searched
  uint8_t tc[66 + 2], beta[64], chroma_scale[70 + 2];
};

template <int MV> __host__ __device__ constexpr int search_smem() {
  return stage_stride<MV>() + 2 * (int)sizeof(SearchWork) + (int)sizeof(SearchShared);
}

// tc / beta of a luma record under one candidate's offsets (LoopFilter.cpp:626-634).
__device__ __forceinline__ EdgeParams luma_edge_apply(uint32_t rec, const SearchShared& sh, int beta_off, int tc_off, int scale) {
  EdgeParams ep;
  const int bs = rec & 3, qp = (int)(int8_t)(rec >> 8);
  ep.bs = bs;
  ep.tc = sh.tc[clip3i(0, 65, qp + 2 * (bs - 1) + 2 * tc_off)] * scale;
  ep.beta = sh.beta[clip3i(0, 63, qp + 2 * beta_off)] * scale;
  ep.no_p = (rec & 4) != 0;
  ep.no_q = (rec & 8) != 0;
  return ep;
}

__device__ __forceinline__ int chroma_edge_tc(uint32_t rec, const SearchShared& sh, int tc_off, int bd_chroma) {
  return sh.tc[clip3i(0, 65, ((int)rec >> 16) + 2 + 2 * tc_off)] * (1 << (bd_chroma - 8));
}

// The chroma filter of one line across an edge (xPelFilterChroma, LoopFilter.cpp:918-957): p1 p0 | q0 q1 -> p0, q0.
__device__ __forceinline__ void filter_chroma_line(int p1, int& p0, int& q0, int q1, int tc, bool no_p, bool no_q, int max_c) {
  const int delta = clip3i(-tc, tc, (((q0 - p0) << 2) + p1 - q1 + 4) >> 3);
  const int np = clip3i(0, max_c, p0 + delta), nq = clip3i(0, max_c, q0 - delta);
  if (!no_p) p0 = np;
  if (!no_q) q0 = nq;
}

__device__ __forceinline__ uint32_t sq_shift(int a, int b, int s) { const int d = a - b; return (uint32_t)(d * d) >> s; }

// Squared differences of a luma task's block (8 rows of 4 samples; row i counts when bit i of `rows`) against the original.
__device__ __forceinline__ uint32_t dist_luma(const uint2 (&r)[8], const uint2 (&o)[8], unsigned rows, int s) {
  uint32_t acc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    if (!((rows >> i) & 1)) continue;
    int a0, a1, a2, a3, b0, b1, b2, b3;
    unpack2(r[i].x, a0, a1); unpack2(r[i].y, a2, a3); unpack2(o[i].x, b0, b1); unpack2(o[i].y, b2, b3);
    acc += sq_shift(a0, b0, s) + sq_shift(a1, b1, s) + sq_shift(a2, b2, s) + sq_shift(a3, b3, s);
  }
  return acc;
}
__device__ __forceinline__ uint32_t dist_chroma(const uint32_t (&r)[8], const uint32_t (&o)[8], unsigned rows, int s) {
  uint32_t acc = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    if (!((rows >> i) & 1)) continue;
    int a0, a1, b0, b1;
    unpack2(r[i], a0, a1); unpack2(o[i], b0, b1);
    acc += sq_shift(a0, b0, s) + sq_shift(a1, b1, s);
  }
  return acc;
}

__device__ __forceinline__ unsigned long long warp_sum(uint32_t v) {
  unsigned long long s = v;
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  return s;
}

// out[slot][candidate][plane]: slot = first_slot + bc.slot[z] (absolute), rows of SEARCH_MAX x 3 words, zeroed by the caller.
template <int MV>
__global__ void __launch_bounds__(SEARCH_THREADS, SEARCH_MIN_CTAS) deblock_search_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc, int num_slots,
                                                                      SearchCands cands, unsigned long long* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int STRIDE = stage_stride<MV>();
  Stage<MV>* const st = reinterpret_cast<Stage<MV>*>(smem);
  SearchWork* const work = reinterpret_cast<SearchWork*>(smem + STRIDE);
  SearchShared& sh = *reinterpret_cast<SearchShared*>(smem + STRIDE + 2 * sizeof(SearchWork));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cw = g.width >> 1;
  const int own0 = g.out_row0 - g.row0, own1 = own0 + g.out_rows;   // held rows whose samples count: all of a whole picture, a band's own
  const int ntx = (g.width + TW - 1) / TW, bands = (g.rows + 4 + TH - 1) / TH;
  const int per_pic = ntx * bands, total = per_pic * num_slots;
  const int K = cands.n;
  int id = blockIdx.x;
  if (id >= total) return;

  // the boxes of `tile` into the stage, all issued by one thread (the K passes over a tile hide the fetch)
  auto issue = [&](int tile) {
    const int z = tile / per_pic, r = tile - z * per_pic, ty = r / ntx, tx = r - ty * ntx;
    const SlotDev& sd = slots[first_slot + bc.slot[z]];
    const bool ctree = sd.info_c != nullptr;
    const int y0 = ty * TH - 4, cy0 = ty * CTH - 2, uy0 = ty * UH - 1;
    ring::mbar_expect_tx(&sh.full, (uint32_t)stage_tx_bytes<MV>(ctree));
    ring::tma_load_3d(&st->y[0][0], &sd.tm_db[0], &sh.full, tx * TW - 8, y0, 0);   // buffer 0: the uploaded picture
    ring::tma_load_3d(&st->c[0][0][0], &sd.tm_db[1], &sh.full, tx * CTW - 8, cy0, 0);
    ring::tma_load_3d(&st->c[1][0][0], &sd.tm_db[2], &sh.full, tx * CTW - 8, cy0, 0);
    ring::tma_load_3d(&st->info[0][0], &sd.tm_info, &sh.full, tx * UW - 4, uy0, 0);
    if (ctree) ring::tma_load_3d(&st->info_c[0][0], &sd.tm_info_c, &sh.full, tx * UW - 4, uy0, 0);
    if (MV == 1) ring::tma_load_3d(&st->mv[0][0], &sd.tm_mv16, &sh.full, (tx * UW - MvBox<1>::OFF) * 2, uy0, 0);
    if (MV == 2) ring::tma_load_3d(&st->mv[0][0], &sd.tm_mv32, &sh.full, (tx * UW - MvBox<2>::OFF) * 4, uy0, 0);
  };
  if (tid == 0) {
    ring::mbar_init(&sh.full, 1);
    ring::mbar_init_fence();
  }
  if (tid < 66) sh.tc[tid] = c_tc[tid];
  if (tid < 64) sh.beta[tid] = c_beta[tid];
  if (tid < 70) sh.chroma_scale[tid] = c_chroma_scale[tid];
  for (int i = tid; i < SEARCH_WARPS_H * SEARCH_MAX * 3; i += SEARCH_THREADS) (&sh.acc[0][0][0])[i] = 0;
  if (tid < SEARCH_WARPS_H * 3) (&sh.common[0][0])[tid] = 0;
  __syncthreads();
  if (tid == 0) issue(id);

  // adds the CTA's sums of slot layer z to the result rows and clears them
  auto flush = [&](int z) {
    __syncthreads();
    unsigned long long* o = out + (size_t)(first_slot + bc.slot[z]) * (SEARCH_MAX * 3);
    for (int i = tid; i < K * 3; i += SEARCH_THREADS) {
      unsigned long long s = 0;
#pragma unroll
      for (int w = 0; w < SEARCH_WARPS_H; w++) { s += (&sh.acc[w][0][0])[i] + sh.common[w][i % 3]; (&sh.acc[w][0][0])[i] = 0; }
      if (s) atomicAdd(o + i, s);
    }
    __syncthreads();
    if (tid < SEARCH_WARPS_H * 3) (&sh.common[0][0])[tid] = 0;   // read again behind at least one more barrier
  };

  const int max_y = (1 << g.bd_luma) - 1, max_c = (1 << g.bd_chroma) - 1, scale_y = 1 << (g.bd_luma - 8);
  const int s_l = cands.shift_luma, s_c = cands.shift_chroma;
  int cur = -1;
  bool ctree = false;
  uint32_t phase = 0;
  for (; id < total; id += gridDim.x) {
    const int z = id / per_pic, r = id - z * per_pic, ty = r / ntx, tx = r - ty * ntx;
    const int next = id + (int)gridDim.x;
    if (z != cur) {   // CTA-uniform
      if (cur >= 0) flush(cur);
      const SlotDev& sd = slots[first_slot + bc.slot[z]];
      for (int i = tid; i < (int)(sizeof(ilf_deblock_params) / 4); i += SEARCH_THREADS) reinterpret_cast<uint32_t*>(&sh.prm)[i] = __ldg(reinterpret_cast<const uint32_t*>(sd.db_params) + i);
      ctree = sd.info_c != nullptr;
      cur = z;
      __syncthreads();
    }
    const int y0 = ty * TH - 4, cy0 = ty * CTH - 2, x0 = tx * TW, cx0 = tx * CTW;
    // this thread's horizontal-pass blocks of the original: the samples the deblocking kernel would store (x < width) in the rows
    // the context owns (a band context deblocks its halo rows too, but they are another band's samples)
    const int u = tid & 31, h = (tid >> 5) & 3;
    const int pl = (tid >> 6) & 1, hc = (tid >> 5) & 1;
    unsigned rows_y = 0, rows_c = 0;
    uint2 org_y[8];
    uint32_t org_c[8];
    if (tid < 128) {
      const SlotDev& sd = slots[first_slot + bc.slot[z]];
      const int x = x0 + 4 * u;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int y = y0 + 8 * h + i;
        const bool in = x < g.width && y >= own0 && y < own1;
        rows_y |= (in ? 1u : 0u) << i;
        org_y[i] = in ? ldg_u2(sd.org[0] + (size_t)y * g.pitch_y + x) : make_uint2(0, 0);
      }
      const int xc = cx0 + 2 * u;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int y = cy0 + 8 * hc + i;
        const bool in = xc < cw && y >= (own0 >> 1) && y < (own1 >> 1);
        rows_c |= (in ? 1u : 0u) << i;
        org_c[i] = in ? __ldg(reinterpret_cast<const uint32_t*>(sd.org[1 + pl] + (size_t)y * g.pitch_c + xc)) : 0u;
      }
    }
    Tile<MV> t;
    t.st = st;
    t.ctree = ctree;
    ring::mbar_wait(&sh.full, phase);
    phase ^= 1u;

    // ---- offset-independent records of this thread's four segments (the task split of deblock_kernel) ----
    const int thr = sh.prm.mv_threshold;
    uint32_t rec_lv = 0, rec_cv = 0, rec_lh = 0, rec_ch = 0;
    const int ev = tid < 128 ? (tid & 15) : 16, sgv = tid < 128 ? (tid >> 4) : tid - 128;    // luma vertical task (tid < 136)
    const int plv = tid < 128 ? (tid >> 6) : ((tid - 128) >> 3), kv = tid < 128 ? ((tid >> 3) & 7) : 8, sgc = tid & 7;   // chroma vertical (tid < 144)
    if (tid < 17 * 8) rec_lv = luma_edge_record(t, thr, sgv, 2 * ev, sgv, 2 * ev - 1, true);
    if (tid < 2 * 9 * 8) rec_cv = chroma_edge_record(t.cinfo(sgc, 4 * kv), t.cinfo(sgc, 4 * kv - 1), sh.prm, sh.chroma_scale, true, plv);
    if (tid < 128) {
      rec_lh = luma_edge_record(t, thr, 2 * h + 1, u, 2 * h, u, false);
      rec_ch = chroma_edge_record(t.cinfo(4 * hc + 1, u), t.cinfo(4 * hc, u), sh.prm, sh.chroma_scale, false, pl);
    }
    if (!__syncthreads_or((int)(rec_lv | rec_cv | rec_lh | rec_ch))) {
      // nothing in the tile is filtered under any candidate: measure the staged samples once
      if (tid < 128) {
        uint2 raw[8];
        uint32_t rc[8];
#pragma unroll
        for (int i = 0; i < 8; i++) {
          raw[i] = *reinterpret_cast<const uint2*>(t.y(8 * h + i, 4 * u));
          rc[i] = *reinterpret_cast<const uint32_t*>(t.ch(pl, 8 * hc + i, 2 * u));
        }
        const unsigned long long dy = warp_sum(dist_luma(raw, org_y, rows_y, s_l)), dc = warp_sum(dist_chroma(rc, org_c, rows_c, s_c));
        if (lane == 0) { sh.common[warp][0] += dy; sh.common[warp][1 + pl] += dc; }
      }
      __syncthreads();   // the stage is free
      if (tid == 0 && next < total) issue(next);
      continue;
    }

    for (int k = 0; k < K; k++) {
      SearchWork* const w = work + (k & 1);
      {
        const uint4* src = reinterpret_cast<const uint4*>(st);
        uint4* dst = reinterpret_cast<uint4*>(w);
        for (int i = tid; i < (int)(sizeof(SearchWork) / 16); i += SEARCH_THREADS) dst[i] = src[i];
      }
      __syncthreads();
      // the records are in registers and the samples in the work buffer: the stage can take the next tile
      if (k == K - 1 && tid == 0 && next < total) issue(next);
      const int beta_off = cands.c[k].beta_offset_div2, tc_off = cands.c[k].tc_offset_div2;

      // ---- vertical edges (deblock_kernel's luma and chroma tasks) ----
      if (rec_lv) {
        const EdgeParams ep = luma_edge_apply(rec_lv, sh, beta_off, tc_off, scale_y);
        int16_t* pp = &w->y[4 * sgv][8 * ev - 4 + 8];
        int16_t* pq = &w->y[4 * sgv][8 * ev + 8];
        int L[4][8];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const uint2 a = *reinterpret_cast<const uint2*>(pp + i * BW), b = *reinterpret_cast<const uint2*>(pq + i * BW);
          unpack2(a.x, L[i][0], L[i][1]); unpack2(a.y, L[i][2], L[i][3]); unpack2(b.x, L[i][4], L[i][5]); unpack2(b.y, L[i][6], L[i][7]);
        }
        if (filter_luma_segment(L, ep, max_y)) {
#pragma unroll
          for (int i = 0; i < 4; i++) {
            *reinterpret_cast<uint2*>(pp + i * BW) = make_uint2(pack2(L[i][0], L[i][1]), pack2(L[i][2], L[i][3]));
            *reinterpret_cast<uint2*>(pq + i * BW) = make_uint2(pack2(L[i][4], L[i][5]), pack2(L[i][6], L[i][7]));
          }
        }
      }
      if (rec_cv) {
        const int tc = chroma_edge_tc(rec_cv, sh, tc_off, g.bd_chroma);
        int16_t* pp = &w->c[plv][2 * sgc][8 * kv - 2 + 8];
        int16_t* pq = &w->c[plv][2 * sgc][8 * kv + 8];
#pragma unroll
        for (int i = 0; i < 2; i++) {
          int p0 = pp[i * BCW + 1], q0 = pq[i * BCW];
          filter_chroma_line(pp[i * BCW], p0, q0, pq[i * BCW + 1], tc, rec_cv & 2, rec_cv & 4, max_c);
          pp[i * BCW + 1] = (int16_t)p0;
          pq[i * BCW] = (int16_t)q0;
        }
      }
      __syncthreads();

      // ---- horizontal edges + distortion of the blocks the deblocking kernel would store ----
      if (tid < 128) {
        uint2 raw[8];
#pragma unroll
        for (int i = 0; i < 8; i++) raw[i] = *reinterpret_cast<const uint2*>(&w->y[8 * h + i][4 * u + 8]);
        if (rec_lh) {
          const EdgeParams ep = luma_edge_apply(rec_lh, sh, beta_off, tc_off, scale_y);
          int L[4][8];
#pragma unroll
          for (int i = 0; i < 8; i++) { unpack2(raw[i].x, L[0][i], L[1][i]); unpack2(raw[i].y, L[2][i], L[3][i]); }
          if (filter_luma_segment(L, ep, max_y)) {
#pragma unroll
            for (int i = 1; i < 7; i++) raw[i] = make_uint2(pack2(L[0][i], L[1][i]), pack2(L[2][i], L[3][i]));
          }
        }
        uint32_t rc[8];
#pragma unroll
        for (int i = 0; i < 8; i++) rc[i] = *reinterpret_cast<const uint32_t*>(&w->c[pl][8 * hc + i][2 * u + 8]);
        if (rec_ch) {
          const int tc = chroma_edge_tc(rec_ch, sh, tc_off, g.bd_chroma);
          int a[4], b[4];
#pragma unroll
          for (int i = 0; i < 4; i++) unpack2(rc[i], a[i], b[i]);
          filter_chroma_line(a[0], a[1], a[2], a[3], tc, rec_ch & 2, rec_ch & 4, max_c);
          filter_chroma_line(b[0], b[1], b[2], b[3], tc, rec_ch & 2, rec_ch & 4, max_c);
          rc[1] = pack2(a[1], b[1]);
          rc[2] = pack2(a[2], b[2]);
        }
        const unsigned long long dy = warp_sum(dist_luma(raw, org_y, rows_y, s_l)), dc = warp_sum(dist_chroma(rc, org_c, rows_c, s_c));
        if (lane == 0) { sh.acc[warp][k][0] += dy; sh.acc[warp][k][1 + pl] += dc; }
      }
      // (no barrier: the next candidate copies into the other work buffer, and the one after it waits behind the next vertical pass)
    }
  }
  flush(cur);
}

}  // namespace

template <int MV>
static void launch_deblock_search_mv(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, const SearchCands& sc,
                                     unsigned long long* out, cudaStream_t st) {
  constexpr int smem = search_smem<MV>();
  static bool attr_set[64] = {};
  once_per_device(attr_set, [&] { cudaFuncSetAttribute(deblock_search_kernel<MV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
  int dev = 0, sms = 0, per_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, deblock_search_kernel<MV>, SEARCH_THREADS, smem);
  const int ntx = (g.width + TW - 1) / TW, bands = (g.rows + 4 + TH - 1) / TH;
  const long long total = (long long)ntx * bands * num_slots;
  const dim3 grid((unsigned)std::min<long long>(total, (long long)std::max(1, sms * per_sm)));
  deblock_search_kernel<MV><<<grid, SEARCH_THREADS, smem, st>>>(g, slots, first_slot, ctl, num_slots, sc, out);
}

// One launch per motion-vector representation present (ilf_api.cu); `out` = result rows of slot 0 of the context.
void launch_deblock_search(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, int mv_mode, const ilf_deblock_candidate* cands,
                           int num_cands, int shift_luma, int shift_chroma, unsigned long long* out, cudaStream_t st) {
  SearchCands sc = {};
  for (int k = 0; k < num_cands; k++) sc.c[k] = cands[k];
  sc.n = num_cands;
  sc.shift_luma = shift_luma;
  sc.shift_chroma = shift_chroma;
  if (mv_mode == 0) launch_deblock_search_mv<0>(g, slots, first_slot, num_slots, ctl, sc, out, st);
  else if (mv_mode == 1) launch_deblock_search_mv<1>(g, slots, first_slot, num_slots, ctl, sc, out, st);
  else launch_deblock_search_mv<2>(g, slots, first_slot, num_slots, ctl, sc, out, st);
}

}  // namespace ilf
