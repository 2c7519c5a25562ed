// ilf_alf.cu -- adaptive loop filter: 4x4 block classification + 7x7/5x5 luma and 5x5 chroma diamond filters (sm_100a).
//
// Replaces AdaptiveLoopFilter::ALFProcess after coefficient reconstruction (AdaptiveLoopFilter.cpp:89-138):
//   deriveClassificationBlk :292-463   Laplacian activity/direction -> classIdx (0..24), transposeIdx (0..3)
//   filterBlk<7/5>          :465-650   point-symmetric diamond FIR, (sum + 256) >> 9, clip to [0, 2^bd - 1]
// The source is the whole SAO'd picture padded by 3 replicated samples (:90-92, Buffer.h:433-465).  CTUs whose enable
// flag is 0 are copied through (the stage reads one buffer and writes the other).
//
// Data movement (both kernels): band walking over a TMA ring (ilf_ring.cuh).  A CTA owns a band of 32 rows of a plane and
// walks it in tiles of TW = 64 samples; the TMA unit delivers each tile with its halo (box 80 x 38 luma, 80 x 36
// chroma) into a ring of shared-memory stages ahead of the arithmetic.  Per tile the CTA builds a work tile: the staged
// tile plus 4 halo columns from the neighbouring tiles of the ring, with the border padding applied (build_work_tile).
//
// Luma, per tile (2 TW = 128 threads, one thread = one 4x4 block from classification to output):
//   phase 1  work tile (int16, two samples per 32-bit word)
//   phase 2  1-D Laplacians two samples per instruction on biased 16-bit lanes, summed per "quad" = 4x4 samples at offset
//            (-2, -2) from the block grid (a task = one quad: two word columns x 4 rows with a rolling 3-row window; the
//            lanes of a quad are folded with IDP.2A against 0x0101)
//   phase 3  a block's 8x8 classification window is exactly 2x2 quads: four 16-byte loads, class + transpose in a register
//   phase 4  each thread filters its block with the (class, transpose) entry of the per-picture table that
//            ilf_set_alf_params precomputed.  Two arithmetic paths, chosen per picture by the host (SlotDev::alf_mode):
//              dot-product path (ilf_alf_tab.cuh): IDP.2A on the packed words of the window, two taps per instruction,
//                nothing unpacked -- 20 instead of ~33 instructions per sample; needs the outer coefficients in int8
//              general path: 32-bit IMAD on unpacked samples with point-symmetric pair sums, any int16 coefficients
// Tiles whose blocks are all in CTUs with ALF off are copied through without classification.
#include "ilf_common.cuh"
#include "ilf_ring.cuh"
#include "ilf_alf_tab.cuh"

namespace ilf {
namespace {

// ---- band walking (ilf_ring.cuh): shared by the chroma kernel (and the luma kernel) ----
constexpr int TW = ALF_TILE;        // tile width in samples
constexpr int BR = ALF_BAND_ROWS;   // rows of a band
constexpr int WP = TW + 16;         // work-tile pitch in samples: [8: left halo slot][128][8: right halo slot], 288-byte rows
constexpr int WX0 = 8;              // work-tile column of the tile's first sample
#ifndef ALF_RING
#define ALF_RING 4
#endif
#ifndef ALF_L_CTAS
#define ALF_L_CTAS (ALF_TILE_W == 128 ? 3 : 5)
#endif
constexpr int RING_STAGES = ALF_RING;  // the tile being filtered + the tiles in flight
constexpr int L_CTAS = ALF_L_CTAS;     // resident luma CTAs per SM the kernel is built for

// A stage of the ring IS the work tile: the TMA box starts 8 samples left of the tile (16-byte aligned) and is WP wide, so
// it carries the tile's horizontal halo with it; these kernels are instruction-bound, the 12.5 % of re-read columns come
// out of L2 and cost nothing.  Out-of-picture samples arrive as zeros; the filters read the picture "padded by
// replication" (AdaptiveLoopFilter.cpp:90-92, Buffer.h:433-465), so tiles that touch a picture border repeat the nearest
// picture sample into the halo: first along the rows (left / right border), then whole rows (top / bottom border).
// vw = valid samples of this tile's rows, ytop = plane row of staged row 0, ph = plane rows.  CTA-uniform; every thread
// of the CTA must call it.
template <int SR, int HALO, int NTHREADS>
__device__ __forceinline__ void pad_borders(int16_t* __restrict__ W, bool left, bool right, int vw, int ytop, int ph) {
  const bool top = ytop < 0, bottom = ytop + SR > ph;
  if (!(left || right || top || bottom)) return;
  if (left || right) {
    for (int r = threadIdx.x; r < SR; r += NTHREADS) {
      int16_t* wrow = W + r * WP;
      if (left) { const uint32_t e = (uint16_t)wrow[WX0]; *reinterpret_cast<uint2*>(wrow + WX0 - 4) = make_uint2(e | (e << 16), e | (e << 16)); }
      if (right) { const uint32_t e = (uint16_t)wrow[WX0 + vw - 1]; *reinterpret_cast<uint2*>(wrow + WX0 + vw) = make_uint2(e | (e << 16), e | (e << 16)); }
    }
    __syncthreads();
  }
  if (top || bottom) {
    const int r_last = ph - 1 - ytop;  // staged row of the last picture row
    for (int i = threadIdx.x; i < 2 * HALO * (WP / 8); i += NTHREADS) {
      const int q = i / (WP / 8), c = i - q * (WP / 8);
      // q < HALO: rows above the picture <- staged row -ytop; else: the HALO rows below the picture <- staged row r_last
      if (q < HALO) { if (top && q < -ytop) *reinterpret_cast<uint4*>(W + q * WP + 8 * c) = *reinterpret_cast<const uint4*>(W + (-ytop) * WP + 8 * c); }
      else if (bottom && r_last + 1 + (q - HALO) < SR) *reinterpret_cast<uint4*>(W + (r_last + 1 + q - HALO) * WP + 8 * c) = *reinterpret_cast<const uint4*>(W + r_last * WP + 8 * c);
    }
    __syncthreads();
  }
}

constexpr int L_SR = BR + 2 * ALF_HALO_Y;                      // 38 staged rows
constexpr int L_STAGE_BYTES = WP * L_SR * 2;                   // 10944 bytes per box
constexpr int L_STAGE_STRIDE = (L_STAGE_BYTES + 127) & ~127;   // TMA destinations are 128-byte aligned
constexpr int QW = TW / 4 + 1, QH = BR / 4 + 1;                // 17 x 9 quads of 4x4 samples, first quad at (x0-2, y0-2)
constexpr int L_CELL_BYTES = 2 * QH * QW * 16;                 // {V, H, D0, D1} sums as 32-bit words, two tiles
constexpr int L_EN_BYTES = 2 * 528;                            // ALF flags of the CTU columns a walk touches (16384 / 32, padded), two CTU rows
constexpr int L_ON_BYTES = 256;                                // per tile of a walk (16384 / 64): ALF on anywhere under it
constexpr int L_SMEM_BYTES = RING_STAGES * L_STAGE_STRIDE + L_CELL_BYTES + RING_STAGES * 8 + L_EN_BYTES + L_ON_BYTES;
constexpr int NT = 2 * TW;                                     // TW / 4 blocks across x 8 block rows
constexpr int BPR = TW / 4;                                    // 4x4 blocks per tile row

// Class of one 4x4 block from its four window sums (AdaptiveLoopFilter.cpp:390-451); the two small tables live in immediates.
__device__ __forceinline__ int classify(int sum_v, int sum_h, int sum_d0, int sum_d1, int shift) {
  const int activity = min(15, (sum_v + sum_h) >> (shift - 5));           // Clip3(0, 15, (tempAct * 32) >> shift), sums are >= 0
  // th[16] = {0, 1, 2, 2, 2, 2, 2, 3, 3, 3, 3, 3, 3, 3, 3, 4} (:294), one nibble per entry
  int class_idx = (int)(((activity & 8) ? 0x43333333u : 0x32222210u) >> (4 * (activity & 7))) & 7;
  int hv1, hv0, d1, d0, dir_hv, dir_d;
  if (sum_v > sum_h) { hv1 = sum_v; hv0 = sum_h; dir_hv = 1; } else { hv1 = sum_h; hv0 = sum_v; dir_hv = 3; }
  if (sum_d0 > sum_d1) { d1 = sum_d0; d0 = sum_d1; dir_d = 0; } else { d1 = sum_d1; d0 = sum_d0; dir_d = 2; }
  int hvd1, hvd0, main_dir, sec_dir;
  // the reference multiplies in `int` and x86 wraps mod 2^32 (:420; SURVEY.md a14): multiply unsigned, compare signed
  if ((int)((unsigned)d1 * (unsigned)hv0) > (int)((unsigned)hv1 * (unsigned)d0)) {
    hvd1 = d1; hvd0 = d0; main_dir = dir_d; sec_dir = dir_hv;
  } else {
    hvd1 = hv1; hvd0 = hv0; main_dir = dir_hv; sec_dir = dir_d;
  }
  int strength = 0;
  if (hvd1 > 2 * hvd0) strength = 1;
  if (hvd1 * 2 > 9 * hvd0) strength = 2;
  if (strength) class_idx += (((main_dir & 1) << 1) + strength) * 5;
  // transposeTable[8] = {0, 1, 0, 2, 2, 3, 1, 3} (:450)
  return class_idx | (int)((0x31322010u >> (4 * (main_dir * 2 + (sec_dir >> 1)))) & 3) << 5;
}

// One work-tile row of a block's window: p = sample x - 4 (8-byte aligned); v[i] = sample x - 4 + i
__device__ __forceinline__ void load_win12(const int16_t* p, int v[12]) {
  const uint2 a = *reinterpret_cast<const uint2*>(p), b = *reinterpret_cast<const uint2*>(p + 4), c = *reinterpret_cast<const uint2*>(p + 8);
  v[0] = a.x & 0xFFFF; v[1] = a.x >> 16; v[2] = a.y & 0xFFFF; v[3] = a.y >> 16;
  v[4] = b.x & 0xFFFF; v[5] = b.x >> 16; v[6] = b.y & 0xFFFF; v[7] = b.y >> 16;
  v[8] = c.x & 0xFFFF; v[9] = c.x >> 16; v[10] = c.y & 0xFFFF; v[11] = c.y >> 16;
}

// IDP.2A: c + a.lo16 * b.byte[0 | 2] + a.hi16 * b.byte[1 | 3]; samples unsigned, coefficients signed
__device__ __forceinline__ int dp2a_lo(uint32_t a, uint32_t b, int c) { int d; asm("dp2a.lo.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ int dp2a_hi(uint32_t a, uint32_t b, int c) { int d; asm("dp2a.hi.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
__device__ __forceinline__ uint32_t dp2a_uu(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }

// Dot-product filter of ONE output sample (ilf_alf_tab.cuh).  R = radius of the slot layout the coefficient words `cw` are in,
// RT = radius of the filter (RT < R: a 5x5 luma filter in the 7x7 layout; its empty slots are skipped at compile time).
// HI_CENTRE: only the centre coefficient has a high part (the usual case: its four neighbours fit int8) -- one IDP instead of four.
// row(dy) gives the packed words of window row y + dy; word m of a row holds the samples at x offsets 2m - XOFF, 2m - XOFF + 1
// from output sample 0 of the thread, j = index of this output sample.  Rows -RT and +RT hold one tap each with the same
// coefficient (point symmetry): top_bottom, when given, is the packed SUM of the two rows and one IDP serves both.
// Everything folds at compile time once unrolled.
template <int R, int RT, int XOFF, bool HI_CENTRE, typename RowFn>
__device__ __forceinline__ int dp_filter_sample(RowFn row, const uint32_t* top_bottom, const uint32_t* cw, int j) {
  const int p = j & 1;
  constexpr int NR = alftab::num_regs<R>();
  int acc = 256, hi = 0;
#pragma unroll
  for (int dy = -RT; dy <= RT; dy++)
#pragma unroll
    for (int q = 0; q <= R; q++) {
      if (!alftab::holds<R, RT>(p, dy, q)) continue;
      if (top_bottom && dy == -RT) continue;
      const int s = alftab::slot<R>(p, dy, q), m = (j + alftab::dx0<R>(p, q) + XOFF) / 2;
      const uint32_t ww = top_bottom && dy == RT ? top_bottom[m] : row(dy)[m];
      acc = (s & 1) ? dp2a_hi(ww, cw[p * NR + (s >> 1)], acc) : dp2a_lo(ww, cw[p * NR + (s >> 1)], acc);
    }
#pragma unroll
  for (int dy = -1; dy <= 1; dy++)
#pragma unroll
    for (int q = 0; q <= 1; q++) {
      if (!alftab::holds<1, 1>(p, dy, q)) continue;
      if (HI_CENTRE && !(dy == 0 && alftab::dx0<1>(p, q) <= 0 && alftab::dx0<1>(p, q) + 1 >= 0)) continue;
      const int s = alftab::slot<1>(p, dy, q);
      const uint32_t ww = row(dy)[(j + alftab::dx0<1>(p, q) + XOFF) / 2];
      hi = (s & 1) ? dp2a_hi(ww, cw[2 * NR + p * 2 + (s >> 1)], hi) : dp2a_lo(ww, cw[2 * NR + p * 2 + (s >> 1)], hi);
    }
  return (acc + (hi << alftab::HI_SHIFT)) >> 9;
}

// Laplacians of one quad: 4x4 samples at (x0 - 2 + 4 qj, y0 - 2 + 4 qi) of a work tile, two samples per instruction.  Reads
// work-tile rows 4 qi .. 4 qi + 5, words 2 + 2 qj .. 5 + 2 qj.  Everything is plain 32-bit arithmetic on biased lanes (no lane
// ever borrows or carries): with K = 2^(bd+1), t' = 2c + K - a - b lies in (0, 2K), and max(t', 2K - t') = K + |2c - a - b|; four
// rows of a lane stay below 2^16 up to 12 bit.  (__vsub2 / __vneg2 and the packed abs-diffs are multi-instruction emulations on
// sm_100a.)  Returns {V, H, D0, D1}: IDP.2A against {1, 1} adds both halves of a word in 32 bits; a quad collected K sixteen times.
__device__ __forceinline__ uint4 lap_quad(const int16_t* W, int qi, int qj, uint32_t lap_k) {
  const uint32_t* wp = reinterpret_cast<const uint32_t*>(W) + (4 * qi) * (WP / 2) + 2 + 2 * qj;
  const uint32_t lap_k2 = lap_k << 1;
  // rows[r][j]: centre / left-shifted / right-shifted word of row r, column j
  uint32_t c[6][2], l[6][2], rr[6][2];
#pragma unroll
  for (int r = 0; r < 6; r++) {
    const uint2 a = *reinterpret_cast<const uint2*>(wp + r * (WP / 2)), b = *reinterpret_cast<const uint2*>(wp + r * (WP / 2) + 2);
    const uint32_t f12 = __funnelshift_r(a.y, b.x, 16);
    c[r][0] = a.y; c[r][1] = b.x; l[r][0] = __funnelshift_r(a.x, a.y, 16); rr[r][0] = f12; l[r][1] = f12; rr[r][1] = __funnelshift_r(b.x, b.y, 16);
  }
  uint32_t acc[4][2];
#pragma unroll
  for (int j = 0; j < 2; j++) {
    uint32_t v[4][4];
#pragma unroll
    for (int r = 1; r <= 4; r++) {
      const uint32_t c2k = c[r][j] + c[r][j] + lap_k;
      uint32_t u;
      u = c2k - c[r - 1][j] - c[r + 1][j]; v[0][r - 1] = __vmaxu2(u, lap_k2 - u);    // K + |2c - up - down|
      u = c2k - l[r][j] - rr[r][j]; v[1][r - 1] = __vmaxu2(u, lap_k2 - u);           // K + |2c - left - right|
      u = c2k - l[r - 1][j] - rr[r + 1][j]; v[2][r - 1] = __vmaxu2(u, lap_k2 - u);   // K + |2c - up-left - down-right|
      u = c2k - rr[r - 1][j] - l[r + 1][j]; v[3][r - 1] = __vmaxu2(u, lap_k2 - u);   // K + |2c - up-right - down-left|
    }
#pragma unroll
    for (int d = 0; d < 4; d++) acc[d][j] = (v[d][0] + v[d][1]) + v[d][2] + v[d][3];
  }
  const uint32_t quad_bias = 0u - ((lap_k & 0xFFFFu) << 4);
  uint4 o;
  o.x = dp2a_uu(acc[0][0], 0x0101u, dp2a_uu(acc[0][1], 0x0101u, quad_bias));
  o.y = dp2a_uu(acc[1][0], 0x0101u, dp2a_uu(acc[1][1], 0x0101u, quad_bias));
  o.z = dp2a_uu(acc[2][0], 0x0101u, dp2a_uu(acc[2][1], 0x0101u, quad_bias));
  o.w = dp2a_uu(acc[3][0], 0x0101u, dp2a_uu(acc[3][1], 0x0101u, quad_bias));
  return o;
}

// Luma block, dot-product path: wp = window row 0 (block row 0 minus 3), sample x - 4; tab = the block's table entry.
template <int RT, bool HI_CENTRE>
__device__ __forceinline__ void filter_block_dp(const int16_t* wp, const uint32_t* __restrict__ tab, int16_t* __restrict__ out, int pitch, int max_val) {
  uint32_t cw[alftab::LUMA_WORDS];
  {
    const uint4* tp = reinterpret_cast<const uint4*>(tab);
#pragma unroll
    for (int i = 0; i < alftab::LUMA_WORDS / 4; i++) { const uint4 v = __ldg(tp + i); cw[4 * i] = v.x; cw[4 * i + 1] = v.y; cw[4 * i + 2] = v.z; cw[4 * i + 3] = v.w; }
  }
  uint32_t w[10][6];  // w[s][m] = samples (x - 4 + 2m, x - 3 + 2m) of window row s
  auto load = [&](int s) {
    const uint2 a = *reinterpret_cast<const uint2*>(wp + s * WP), b = *reinterpret_cast<const uint2*>(wp + s * WP + 4), c = *reinterpret_cast<const uint2*>(wp + s * WP + 8);
    w[s][0] = a.x; w[s][1] = a.y; w[s][2] = b.x; w[s][3] = b.y; w[s][4] = c.x; w[s][5] = c.y;
  };
#pragma unroll
  for (int s = 3 - RT; s < 3 + RT; s++) load(s);
#pragma unroll
  for (int o = 0; o < 4; o++) {
    load(o + 3 + RT);
    uint32_t tbsum[6];  // rows -RT and +RT: one tap each (dx = 0, words 2 and 3), same coefficient
    tbsum[2] = w[o + 3 - RT][2] + w[o + 3 + RT][2];
    tbsum[3] = w[o + 3 - RT][3] + w[o + 3 + RT][3];
    int r[4];
#pragma unroll
    for (int j = 0; j < 4; j++) r[j] = __vimin_s32_relu(dp_filter_sample<3, RT, 4, HI_CENTRE>([&](int dy) { return w[o + 3 + dy]; }, tbsum, cw, j), max_val);
    *reinterpret_cast<uint2*>(out + (size_t)o * pitch) = make_uint2(__byte_perm(r[0], r[1], 0x5410), __byte_perm(r[2], r[3], 0x5410));
  }
}

// Luma CTA: band blockIdx.y, horizontal segment blockIdx.x of nseg.  Per tile: Laplacians of the tile's 17 x 9 quads (phase 2), ONE CTA
// barrier, then every thread classifies and filters its 4x4 block (phases 3, 4).  The quads are double-buffered, so the barrier of
// tile t + 1 is also what tells thread 0 that the stage of tile t is free again.
//
// What bounds this kernel (tools/ubench/rf.cu, mix.cu; profiles/r02_alf_*): IDP.2A issues every second clock on the one heavy
// FMA pipe, and an ALU-pipe instruction issued between two IDPs still costs 0.5 - 1 clock (a 1:1 mix of IDP and IADD3 / VIMNMX /
// SHF / PRMT with register operands runs at 0.63 - 0.73 instructions per clock, not 1.0), so interleaving the phases buys
// nothing: time = 2 x IDPs + ~0.8 x everything else, and the work is cut by instruction count: 16 IDP per sample (15 low parts
// + the centre's high part), Laplacians two samples per instruction, per-tile bookkeeping kept out of the loop.
template <bool CLASSIFY_ONLY>
__device__ __forceinline__ void alf_luma_cta(unsigned char* smem, const Geom& g, const SlotDev& sd, unsigned ctl, int nseg) {
  if (ctl_skip(ctl, 0) || (int)blockIdx.x >= nseg) return;
  const int tid = threadIdx.x;
  const int rows = g.rows;
  const int ntx = (g.width + TW - 1) / TW;
  const int ta = (int)blockIdx.x * ntx / nseg, tb = ((int)blockIdx.x + 1) * ntx / nseg;
  if (ta >= tb) return;
  uint4(*quad_buf)[QH][QW] = reinterpret_cast<uint4(*)[QH][QW]>(smem + RING_STAGES * L_STAGE_STRIDE);  // {V, H, D0, D1} per quad, two tiles
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + RING_STAGES * L_STAGE_STRIDE + L_CELL_BYTES);
  uint8_t* en_s = smem + RING_STAGES * L_STAGE_STRIDE + L_CELL_BYTES + RING_STAGES * 8;  // ALF flag of the CTUs of this band's CTU row, from column c0
  uint8_t* on_s = en_s + L_EN_BYTES;                                                      // per tile of the walk: ALF on in any CTU under it
  const int y0 = (int)blockIdx.y * BR;  // local rows
  const int src_buf = ctl_src(ctl, 0);
  const CUtensorMap* map = &sd.tm_alf[0];
  auto issue = [&](int t, int stage) {
    ring::mbar_expect_tx(&full[stage], L_STAGE_BYTES);
    ring::tma_load_3d(smem + stage * L_STAGE_STRIDE, map, &full[stage], t * TW - WX0, y0 - ALF_HALO_Y, src_buf);
  };
  if (tid == 0) {
    for (int i = 0; i < RING_STAGES; i++) ring::mbar_init(&full[i], 1);
    ring::mbar_init_fence();
    pdl_wait();  // the stage before this one has written the planes read from here on
    for (int i = 0; i < RING_STAGES && ta + i < tb; i++) issue(ta + i, i);
  }
  // this thread's 4x4 block of every tile: BPR blocks across, 8 block rows
  const int bj = tid % BPR, bi = tid / BPR;
  const int by = y0 + 4 * bi;
  const int c0 = (ta * TW) >> g.ctu_log2, c1 = min(g.ctus_w - 1, (tb * TW - 1) >> g.ctu_log2);  // CTU columns this walk touches
  // A band of 32 rows lies in one CTU row of a whole picture; in a band context the held rows start 16 rows above a CTU row, so
  // it can straddle two.  en_s[r][c]: flags of CTU row r0 + r, columns from c0.
  const int r0 = (y0 + g.row0) >> g.ctu_log2, r1 = min(g.ctus_h - 1, (min(y0 + BR, rows) - 1 + g.row0) >> g.ctu_log2);
  const int ncol = c1 - c0 + 1;
  if (!CLASSIFY_ONLY) {
    for (int i = tid; i < (r1 - r0 + 1) * ncol; i += NT) en_s[i] = sd.alf_ctu_enable[(size_t)(r0 + i / ncol) * g.ctus_w + c0 + i % ncol];
    for (int t = ta + tid; t < tb; t += NT) {
      bool any = false;
      for (int r = r0; r <= r1; r++)
        for (int c = (t * TW) >> g.ctu_log2; c <= min(c1, (t * TW + TW - 1) >> g.ctu_log2); c++) any |= sd.alf_ctu_enable[(size_t)r * g.ctus_w + c] != 0;
      on_s[t - ta] = any;
    }
  }
  const int en_off = (min(r1, (by + g.row0) >> g.ctu_log2) - r0) * ncol - c0;   // this thread's row of en_s
  int16_t* __restrict__ dst = sd.buf[ctl_dst(ctl, 0)][0];
  const int max_val = (1 << g.bd_luma) - 1;
  const bool is7 = CLASSIFY_ONLY ? true : (ctl & CTL_ALF_7X7) != 0;
  const bool dot = CLASSIFY_ONLY ? false : (ctl & CTL_ALF_DOT_Y) != 0;  // dot-product path (ilf_alf_tab.cuh), else the general path
  const bool hi_centre = (ctl & CTL_ALF_HIC_Y) != 0;                    // only the centre coefficient has a high part
  const int shift = g.bd_luma + 4;
  const uint32_t lap_k = 0x10001u << (g.bd_luma + 1);  // Laplacian lane bias K in both lanes
  const bool vborder = y0 - ALF_HALO_Y < 0 || y0 - ALF_HALO_Y + L_SR > rows;
  // the quads of this thread: one, and for 25 threads of the last warp a second one
  const int qi0 = tid / QW, qj0 = tid % QW, qi1 = (tid - 96 + NT) / QW, qj1 = (tid - 96 + NT) % QW;
  const bool two_quads = tid >= 96 && tid - 96 + NT < QW * QH;
  __syncthreads();  // barriers initialised, flags staged
  pdl_wait();  // every thread: this kernel's stores must not overtake the previous stage's reads either

  int stage = 0;
  uint32_t parity = 0;
  int16_t* out = dst + (size_t)by * g.pitch_y + ta * TW + 4 * bj;
  for (int tx = ta; tx < tb; tx++, out += TW) {
    ring::mbar_wait(&full[stage], parity);
    const bool on = CLASSIFY_ONLY || on_s[tx - ta] != 0;   // CTA-uniform: ALF on in some CTU under this tile
    int16_t* W = reinterpret_cast<int16_t*>(smem + stage * L_STAGE_STRIDE);
    uint4(*quad)[QW] = quad_buf[(tx - ta) & 1];
    if (on) {
      // ---- phase 1: the stage is the work tile; border tiles get their padding ----
      if (vborder || tx == 0 || tx == ntx - 1) pad_borders<L_SR, ALF_HALO_Y, NT>(W, tx == 0, tx == ntx - 1, min(TW, g.width - tx * TW), y0 - ALF_HALO_Y, rows);
      // ---- phase 2: Laplacians per quad ----
      quad[qi0][qj0] = lap_quad(W, qi0, qj0, lap_k);
      if (two_quads) quad[qi1][qj1] = lap_quad(W, qi1, qj1, lap_k);
    }
    __syncthreads();  // quads of this tile complete; every thread has finished the previous tile
    if (tid == 0 && tx > ta && tx - 1 + RING_STAGES < tb) issue(tx - 1 + RING_STAGES, stage == 0 ? RING_STAGES - 1 : stage - 1);
    const int bx = tx * TW + 4 * bj;
    const bool blk_in = bx < g.width && by < rows;
    if (!on) {
      // every CTU under this tile has ALF off: copy through
      if (blk_in) {
#pragma unroll
        for (int o = 0; o < 4; o++) *reinterpret_cast<uint2*>(out + (size_t)o * g.pitch_y) = *reinterpret_cast<const uint2*>(W + (ALF_HALO_Y + 4 * bi + o) * WP + WX0 + 4 * bj);
      }
    } else {
      // ---- phase 3: the block's 8x8 window = quads (bi, bj) .. (bi + 1, bj + 1) -> class ----
      const uint4 q00 = quad[bi][bj], q01 = quad[bi][bj + 1], q10 = quad[bi + 1][bj], q11 = quad[bi + 1][bj + 1];
      const int sv = (int)(q00.x + q01.x + q10.x + q11.x), sh = (int)(q00.y + q01.y + q10.y + q11.y);
      const int sd0 = (int)(q00.z + q01.z + q10.z + q11.z), sd1 = (int)(q00.w + q01.w + q10.w + q11.w);
      const int cl = classify(sv, sh, sd0, sd1, shift);
      if (CLASSIFY_ONLY) {
        if (blk_in) sd.alf_class[(size_t)(by >> 2) * g.units_w + (bx >> 2)] = (uint8_t)cl;
      } else if (blk_in) {
        // ---- phase 4: filter the block ----
        const int16_t* wp = W + (4 * bi) * WP + WX0 + 4 * bj - 4;  // window row 0 (= block row 0 minus 3), sample x - 4
        if (en_s[en_off + (bx >> g.ctu_log2)] == 0) {
#pragma unroll
          for (int o = 0; o < 4; o++) *reinterpret_cast<uint2*>(out + (size_t)o * g.pitch_y) = *reinterpret_cast<const uint2*>(wp + (3 + o) * WP + 4);
        } else if (dot) {
          const uint32_t* tab = sd.alf_coef_dp + ((cl & 31) * 4 + (cl >> 5)) * alftab::LUMA_WORDS;
          if (is7) {
            if (hi_centre) filter_block_dp<3, true>(wp, tab, out, g.pitch_y, max_val);
            else filter_block_dp<3, false>(wp, tab, out, g.pitch_y, max_val);
          } else {
            if (hi_centre) filter_block_dp<2, true>(wp, tab, out, g.pitch_y, max_val);
            else filter_block_dp<2, false>(wp, tab, out, g.pitch_y, max_val);
          }
        } else {
          int f[16];
          {
            const int4* cp = reinterpret_cast<const int4*>(sd.alf_coef + ((cl & 31) * 4 + (cl >> 5)) * 16);
            const int4 a = __ldg(cp), b = __ldg(cp + 1), c = __ldg(cp + 2), d = __ldg(cp + 3);
            f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
            f[8] = c.x; f[9] = c.y; f[10] = c.z; f[11] = c.w; f[12] = d.x; f[13] = d.y; f[14] = d.z; f[15] = d.w;
          }
          // w[s][i] = sample (x - 4 + i, y - 3 + s); output sample j of output row o reads w[o + 3 + dy][j + 4 + dx]
          int w[10][12];
          if (is7) {
#pragma unroll
            for (int s = 0; s < 6; s++) load_win12(wp + s * WP, w[s]);
#pragma unroll
            for (int o = 0; o < 4; o++) {
              load_win12(wp + (o + 6) * WP, w[o + 6]);
              const int(&r0)[12] = w[o + 3];
              int sum[4];
#pragma unroll
              for (int j = 0; j < 4; j++) {
                sum[j] = 256 + f[12] * r0[j + 4] + f[11] * (r0[j + 5] + r0[j + 3]) + f[10] * (r0[j + 6] + r0[j + 2]) + f[9] * (r0[j + 7] + r0[j + 1]);
                sum[j] += f[4] * (w[o + 4][j + 6] + w[o + 2][j + 2]) + f[5] * (w[o + 4][j + 5] + w[o + 2][j + 3]) + f[6] * (w[o + 4][j + 4] + w[o + 2][j + 4]) +
                          f[7] * (w[o + 4][j + 3] + w[o + 2][j + 5]) + f[8] * (w[o + 4][j + 2] + w[o + 2][j + 6]);
                sum[j] += f[1] * (w[o + 5][j + 5] + w[o + 1][j + 3]) + f[2] * (w[o + 5][j + 4] + w[o + 1][j + 4]) + f[3] * (w[o + 5][j + 3] + w[o + 1][j + 5]);
                sum[j] += f[0] * (w[o + 6][j + 4] + w[o][j + 4]);
                sum[j] = __vimin_s32_relu(sum[j] >> 9, max_val);
              }
              const uint32_t p0 = __byte_perm(sum[0], sum[1], 0x5410);
              const uint32_t p1 = __byte_perm(sum[2], sum[3], 0x5410);
              *reinterpret_cast<uint2*>(out + (size_t)o * g.pitch_y) = make_uint2(p0, p1);
            }
          } else {
#pragma unroll
            for (int s = 1; s < 5; s++) load_win12(wp + s * WP, w[s]);
#pragma unroll
            for (int o = 0; o < 4; o++) {
              load_win12(wp + (o + 5) * WP, w[o + 5]);
              const int(&r0)[12] = w[o + 3];
              int sum[4];
#pragma unroll
              for (int j = 0; j < 4; j++) {
                sum[j] = 256 + f[6] * r0[j + 4] + f[5] * (r0[j + 5] + r0[j + 3]) + f[4] * (r0[j + 6] + r0[j + 2]);
                sum[j] += f[1] * (w[o + 4][j + 5] + w[o + 2][j + 3]) + f[2] * (w[o + 4][j + 4] + w[o + 2][j + 4]) + f[3] * (w[o + 4][j + 3] + w[o + 2][j + 5]);
                sum[j] += f[0] * (w[o + 5][j + 4] + w[o + 1][j + 4]);
                sum[j] = __vimin_s32_relu(sum[j] >> 9, max_val);
              }
              const uint32_t p0 = __byte_perm(sum[0], sum[1], 0x5410);
              const uint32_t p1 = __byte_perm(sum[2], sum[3], 0x5410);
              *reinterpret_cast<uint2*>(out + (size_t)o * g.pitch_y) = make_uint2(p0, p1);
            }
          }
        }
      }
    }
    if (++stage == RING_STAGES) { stage = 0; parity ^= 1; }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Chroma: 5x5 diamond, one filter per picture, no classification (filterBlk<ALF_FILTER_5>, AdaptiveLoopFilter.cpp:465-650).
// Band walking over a TMA ring: box (TW + 16) x 36 (2 halo rows each side); a thread filters 8 samples x 2 rows from the work
// tile: 6 window rows of 12 samples are unpacked once into registers and serve both output rows.
// ---------------------------------------------------------------------------------------------------------
constexpr int C_SR = BR + 2 * ALF_HALO_C;
constexpr int C_STAGE_BYTES = WP * C_SR * 2;
static_assert(C_STAGE_BYTES % 128 == 0, "TMA destinations are 128-byte aligned");
constexpr int C_SMEM_BYTES = RING_STAGES * C_STAGE_BYTES + RING_STAGES * 8;
constexpr int NTC = 2 * TW;   // TW / 8 eight-sample groups across x 16 row pairs

// p points at sample x of a work-tile row; v[i] = sample x - 2 + i, i = 0..11
__device__ __forceinline__ void load_row12(const int16_t* p, int v[12]) {
  const uint32_t a = *reinterpret_cast<const uint32_t*>(p - 2);
  const uint4 b = *reinterpret_cast<const uint4*>(p);
  const uint32_t c = *reinterpret_cast<const uint32_t*>(p + 8);
  v[0] = a & 0xFFFF; v[1] = a >> 16;
  v[2] = b.x & 0xFFFF; v[3] = b.x >> 16; v[4] = b.y & 0xFFFF; v[5] = b.y >> 16; v[6] = b.z & 0xFFFF; v[7] = b.z >> 16; v[8] = b.w & 0xFFFF; v[9] = b.w >> 16;
  v[10] = c & 0xFFFF; v[11] = c >> 16;
}

// Chroma, dot-product path: 8 samples x 2 rows per thread from the packed words of a 6-row window (w[r][m] = samples (x - 2 + 2m, x - 1 + 2m)
// of window row r); cw = the picture's chroma filter in the radius-2 layout (ilf_alf_tab.cuh).  9 IDP per sample (8 low parts -- the
// top and bottom rows share one -- and the centre's high part) against 7 IMAD + 6 adds + 4.5 unpacks of the general path.
template <bool HI_CENTRE>
__device__ __forceinline__ void filter_chroma_dp(const int16_t* wp, const uint32_t (&cw)[alftab::CHROMA_WORDS], int16_t* __restrict__ out, int pitch, int nrows, int max_val) {
  uint32_t w[6][6];
#pragma unroll
  for (int r = 0; r < 6; r++) {
    const uint4 b = *reinterpret_cast<const uint4*>(wp + r * WP);
    w[r][0] = *reinterpret_cast<const uint32_t*>(wp + r * WP - 2); w[r][1] = b.x; w[r][2] = b.y; w[r][3] = b.z; w[r][4] = b.w;
    w[r][5] = *reinterpret_cast<const uint32_t*>(wp + r * WP + 8);
  }
#pragma unroll
  for (int o = 0; o < 2; o++) {
    if (o >= nrows) break;
    uint32_t tbsum[6];
#pragma unroll
    for (int m = 1; m <= 4; m++) tbsum[m] = w[o][m] + w[o + 4][m];   // rows -2 and +2: one tap each (dx = 0), same coefficient
    int r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = __vimin_s32_relu(dp_filter_sample<2, 2, 2, HI_CENTRE>([&](int dy) { return w[o + 2 + dy]; }, tbsum, cw, j), max_val);
    *reinterpret_cast<uint4*>(out + (size_t)o * pitch) =
        make_uint4(__byte_perm(r[0], r[1], 0x5410), __byte_perm(r[2], r[3], 0x5410), __byte_perm(r[4], r[5], 0x5410), __byte_perm(r[6], r[7], 0x5410));
  }
}

// Chroma CTA: band `cband` (0 .. 2 bands_c - 1: Cb bands, then Cr bands), horizontal segment blockIdx.x of nseg.
__device__ __forceinline__ void alf_chroma_cta(unsigned char* smem, const Geom& g, const SlotDev& sd, unsigned ctl, int cband, int bands_c, int nseg) {
  const int plane = 1 + (cband >= bands_c), band = cband - (plane - 1) * bands_c;
  if (ctl_skip(ctl, plane) || (int)blockIdx.x >= nseg) return;
  const int tid = threadIdx.x;
  const int cw = g.width >> 1, crows = g.rows >> 1;
  const int ntx = (cw + TW - 1) / TW;
  const int ta = (int)blockIdx.x * ntx / nseg, tb = ((int)blockIdx.x + 1) * ntx / nseg;
  if (ta >= tb) return;
  ring::Walk<RING_STAGES> walk;
  walk.first = ta; walk.last = tb - 1;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + RING_STAGES * C_STAGE_BYTES);
  const int by0 = band * BR;
  const int src_buf = ctl_src(ctl, plane);
  int16_t* __restrict__ dst = sd.buf[ctl_dst(ctl, plane)][plane];
  const CUtensorMap* map = &sd.tm_alf[plane];
  auto stage_ptr = [&](int t) { return reinterpret_cast<int16_t*>(smem + walk.stage(t) * C_STAGE_BYTES); };
  auto issue = [&](int t) {
    uint64_t* bar = &full[walk.stage(t)];
    ring::mbar_expect_tx(bar, C_STAGE_BYTES);
    ring::tma_load_3d(stage_ptr(t), map, bar, t * TW - WX0, by0 - ALF_HALO_C, src_buf);
  };
  if (tid == 0) {
    for (int i = 0; i < RING_STAGES; i++) ring::mbar_init(&full[i], 1);
    ring::mbar_init_fence();
  }
  __syncthreads();
  pdl_wait();  // the stage before this one has written the planes read from here on
  if (tid == 0)
    for (int t = walk.first; t <= walk.last && t < walk.first + RING_STAGES; t++) issue(t);

  int f[7];
#pragma unroll
  for (int i = 0; i < 7; i++) f[i] = sd.alf->chroma_coeff[i];
  const bool dot = (ctl & CTL_ALF_DOT_C) != 0, hi_centre = (ctl & CTL_ALF_HIC_C) != 0;   // dot-product path (ilf_alf_tab.cuh), else the general path
  uint32_t ccw[alftab::CHROMA_WORDS];
  if (dot) {
    const uint4* tp = reinterpret_cast<const uint4*>(sd.alf_coef_dp + 25 * 4 * alftab::LUMA_WORDS);
#pragma unroll
    for (int i = 0; i < alftab::CHROMA_WORDS / 4; i++) { const uint4 v = __ldg(tp + i); ccw[4 * i] = v.x; ccw[4 * i + 1] = v.y; ccw[4 * i + 2] = v.z; ccw[4 * i + 3] = v.w; }
  }
  const int max_val = (1 << g.bd_chroma) - 1;
  const int k = tid % (TW / 8), rg = tid / (TW / 8);  // 8 samples at column 8k, rows 2rg and 2rg + 1 of the band
  const int y = by0 + 2 * rg;
  const uint8_t* __restrict__ en_row = sd.alf_ctu_enable + (size_t)plane * g.ctus_w * g.ctus_h + (size_t)((((y << 1) + g.row0) >> g.ctu_log2) * g.ctus_w);

  for (int tx = ta; tx < tb; tx++) {
    ring::mbar_wait(&full[walk.stage(tx)], walk.parity(tx));
    const int x0 = tx * TW, x = x0 + 8 * k;
    const bool in = x < cw && y < crows;
    const bool en = in && en_row[(x << 1) >> g.ctu_log2] != 0;
    int16_t* W = stage_ptr(tx);
    int16_t* out = dst + (size_t)y * g.pitch_c + x;
    const int nrows = min(2, crows - y);
    if (!__syncthreads_or(en)) {
      // every CTU under this tile has chroma ALF off: copy through
      if (in) {
#pragma unroll
        for (int o = 0; o < 2; o++)
          if (o < nrows) *reinterpret_cast<uint4*>(out + (size_t)o * g.pitch_c) = *reinterpret_cast<const uint4*>(W + (ALF_HALO_C + 2 * rg + o) * WP + WX0 + 8 * k);
      }
    } else {
      pad_borders<C_SR, ALF_HALO_C, NTC>(W, tx == 0, tx == ntx - 1, min(TW, cw - x0), by0 - ALF_HALO_C, crows);
      if (in) {
        const int16_t* wp = W + (2 * rg) * WP + WX0 + 8 * k;  // window row 0 (= output row 0 minus 2), sample x
        if (!en) {
#pragma unroll
          for (int o = 0; o < 2; o++)
            if (o < nrows) *reinterpret_cast<uint4*>(out + (size_t)o * g.pitch_c) = *reinterpret_cast<const uint4*>(wp + (2 + o) * WP);
        } else if (dot) {
          if (hi_centre) filter_chroma_dp<true>(wp, ccw, out, g.pitch_c, nrows, max_val);
          else filter_chroma_dp<false>(wp, ccw, out, g.pitch_c, nrows, max_val);
        } else {
          int w[6][12];
#pragma unroll
          for (int r = 0; r < 6; r++) load_row12(wp + r * WP, w[r]);
#pragma unroll
          for (int o = 0; o < 2; o++) {
            if (o >= nrows) break;
            uint32_t pk2[4];
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
              int sm[2];
#pragma unroll
              for (int h = 0; h < 2; h++) {
                const int j = 2 * jj + h + 2;  // window index of the output sample
                int sum = 256 + f[6] * w[o + 2][j] + f[5] * (w[o + 2][j + 1] + w[o + 2][j - 1]) + f[4] * (w[o + 2][j + 2] + w[o + 2][j - 2]);
                sum += f[1] * (w[o + 3][j + 1] + w[o + 1][j - 1]) + f[2] * (w[o + 3][j] + w[o + 1][j]) + f[3] * (w[o + 3][j - 1] + w[o + 1][j + 1]);
                sum += f[0] * (w[o + 4][j] + w[o][j]);
                sm[h] = __vimin_s32_relu(sum >> 9, max_val);  // clip to [0, max]
              }
              pk2[jj] = __byte_perm(sm[0], sm[1], 0x5410);
            }
            *reinterpret_cast<uint4*>(out + (size_t)o * g.pitch_c) = make_uint4(pk2[0], pk2[1], pk2[2], pk2[3]);
          }
        }
      }
    }
    __syncthreads();  // the stage is free
    if (tid == 0 && tx + RING_STAGES <= walk.last) issue(tx + RING_STAGES);
  }
}

// One launch for the whole ALF stage: grid rows [0, bands_y) are luma bands, [bands_y, bands_y + 2 bands_c) chroma bands.
// The instruction-bound luma CTAs and the memory-bound chroma CTAs share the SMs instead of running back to back.
__global__ void __launch_bounds__(NT, L_CTAS) alf_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc, int bands_y, int bands_c, int nseg_y, int nseg_c) {
  extern __shared__ __align__(128) unsigned char smem[];
  pdl_launch_dependents();
  const SlotDev& sd = slots[first_slot + bc.slot[blockIdx.z]];
  const unsigned ctl = bc.v[blockIdx.z];
  if ((int)blockIdx.y < bands_y) alf_luma_cta<false>(smem, g, sd, ctl, nseg_y);
  else alf_chroma_cta(smem, g, sd, ctl, (int)blockIdx.y - bands_y, bands_c, nseg_c);
}
__global__ void __launch_bounds__(NT, L_CTAS) alf_classify_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc, int nseg) {
  extern __shared__ __align__(128) unsigned char smem[];
  pdl_launch_dependents();
  alf_luma_cta<true>(smem, g, slots[first_slot + bc.slot[blockIdx.z]], bc.v[blockIdx.z], nseg);
}
static_assert(NT == NTC, "luma and chroma CTAs share one launch");

}  // namespace

static int alf_nseg(int bands_total, int ntx, bool luma) {
  if (luma) return pick_segments(bands_total, ntx, 148 * L_CTAS);
  int nseg = (148 * L_CTAS + bands_total - 1) / bands_total;
  return nseg < 1 ? 1 : (nseg > ntx ? ntx : nseg);
}

// The slots' control words say which planes of which slot really run.
void launch_alf(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st) {
  static bool attr_set[64] = {};
  static const int pad = env_int("ILF_ALF_SMEM_PAD");
  const int smem = (L_SMEM_BYTES > C_SMEM_BYTES ? L_SMEM_BYTES : C_SMEM_BYTES) + pad;
  once_per_device(attr_set, [&] { cudaFuncSetAttribute(alf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); });
  const int bands_y = (g.rows + BR - 1) / BR, bands_c = (g.rows / 2 + BR - 1) / BR;
  const int nseg_y = alf_nseg(bands_y * num_slots, (g.width + TW - 1) / TW, true);
  const int nseg_c = alf_nseg(2 * bands_c * num_slots, (g.width / 2 + TW - 1) / TW, false);
  launch_pdl(alf_kernel, dim3(nseg_y > nseg_c ? nseg_y : nseg_c, bands_y + 2 * bands_c, num_slots), dim3(NT), smem, st, g, slots, first_slot, ctl, bands_y,
             bands_c, nseg_y, nseg_c);
}

void launch_alf_classify(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st) {
  static bool attr_set[64] = {};
  once_per_device(attr_set, [&] { cudaFuncSetAttribute(alf_classify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L_SMEM_BYTES); });
  const int bands_y = (g.rows + BR - 1) / BR;
  const int nseg = alf_nseg(bands_y * num_slots, (g.width + TW - 1) / TW, true);
  launch_pdl(alf_classify_kernel, dim3(nseg, bands_y, num_slots), dim3(NT), L_SMEM_BYTES, st, g, slots, first_slot, ctl, nseg);
}

}  // namespace ilf
