// ilf_alf_stats.cu -- encoder ALF statistics on the device-resident picture (sm_100a).
//
// Replaces EncAdaptiveLoopFilter::deriveStatsForFiltering / getBlkStats / calcCovariance
// (source/Lib/EncoderLib/EncAdaptiveLoopFilter.cpp:1317-1514), the largest in-loop cost of the encoder: per CTU and class the
// covariance E[k][l] of the 13 symmetric tap sums of the reconstruction around every sample (7x7 shape), their correlation y[k]
// with (original - reconstruction) and its energy.  The reference accumulates doubles that hold exact integers below 2^53;
// int64 here is bit-equivalent.  Only the 7x7 shape is computed for luma: the 5x5 shape's taps are a subset of it under every
// transposition, so its statistics are rows / columns {2, 5, 6, 7, 10, 11, 12} of the 7x7 record (the host shim slices them).
//
// One thread = one 4x4 block (one class, one transposition): the picture strip is staged in shared memory with its border
// replicated (recYuv.extendBorderPel, :252), the thread walks its 16 samples in the block's TRANSPOSED coordinate frame, so the
// same code serves all four transpositions, forms the 13 tap sums of a sample and adds their 91 + 13 + 1 products to int32
// registers (16 samples of a 12-bit picture stay below 2^31).  The 105 sums of the block then take three steps to the CTU's record
// of its class: (1) a warp whose 32 blocks all share (CTU, class) adds its sums with REDUX (two 16-bit halves, so nothing
// overflows), (2) the result -- in a mixed warp every lane's own sums -- is added to the CTA's accumulators in shared memory (64-bit
// as a low and a high word: 64-bit shared atomics are CAS loops on sm_100a, 32-bit ones are native), (3) after a barrier the
// non-zero accumulators go to L2 with one 64-bit reduction each.  A CTA sends a few hundred reductions instead of 105 per block
// (26 880), which is what bounded the first version of this kernel (14 ms for the luma planes of 17 4K pictures).
// A band context measures its own rows: tiles start at its first own row, border clamps and CTU records use picture coordinates,
// plane rows are addressed from the first held row.  The strip reaches 3 rows (chroma 2) beyond the own rows, inside the halo.
#include <algorithm>
#include "ilf_common.cuh"

namespace ilf {
namespace {

constexpr int ST_W = 128, ST_H = 16;   // luma samples a CTA covers (chroma: the same numbers on a chroma plane); 128 threads, three CTAs per SM
constexpr int NT = (ST_W / 4) * (ST_H / 4);

template <int HALF>
struct Shape {
  static constexpr int N = HALF == 3 ? 13 : 7;
  static constexpr int WORDS = N * (N + 1) / 2 + N + 1;
};

// canonical tap offsets (a, b) of coefficient k, transposeIdx 0: rows -HALF .. -1 left to right, then the left half of the centre row
template <int HALF>
__device__ __forceinline__ void tap_ab(int k, int& a, int& b) {
  int i = 0;
#pragma unroll
  for (int bb = -HALF; bb <= 0; bb++)
#pragma unroll
    for (int aa = -(HALF + bb); aa <= (bb < 0 ? HALF + bb : -1); aa++, i++)
      if (i == k) { a = aa; b = bb; }
}

template <int HALF, bool CLASSES>
__global__ void __launch_bounds__(NT, 3) alf_stats_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc, int plane) {
  constexpr int N = Shape<HALF>::N, WORDS = Shape<HALF>::WORDS;
  // The strip with its halo, staged from 8 samples left of it (16-byte aligned chunks): tile column j = plane column x0 - 8 + j.
  constexpr int TP = ST_W + 16, CH = TP / 8, TR = ST_H + 2 * HALF;
  __shared__ __align__(16) int16_t tile[TR * TP];
  __shared__ __align__(16) int16_t sorg[ST_H * ST_W];   // the source picture's strip
  extern __shared__ uint32_t sacc[];   // [sets][classes][WORDS] low words, then the same number of high words
  const SlotDev& sd = slots[first_slot + bc.slot[blockIdx.z]];
  const unsigned ctl = bc.v[blockIdx.z];
  const int sh = plane ? 1 : 0;
  const int w = g.width >> sh, h = g.height >> sh, pitch = plane ? g.pitch_c : g.pitch_y;
  const int r0 = g.row0 >> sh, yend = (g.out_row0 + g.out_rows) >> sh;   // first held row, end of the own rows (picture rows)
  const int16_t* __restrict__ rec = sd.buf[ctl_src(ctl, plane)][plane];
  const int16_t* __restrict__ org = sd.org[plane];
  const int x0 = blockIdx.x * ST_W, y0 = (g.out_row0 >> sh) + blockIdx.y * ST_H;
  const int ctu_log2 = g.ctu_log2 - sh;
  // CTUs under this tile: sets_x across, sets_y down (1 x 1 for the 128-sample CTUs of the reference's configurations)
  const int sets_x = max(1, ST_W >> ctu_log2), sets_y = max(1, ST_H >> ctu_log2);
  const int num_acc = sets_x * sets_y * (CLASSES ? 25 : 1) * WORDS;
  for (int i = threadIdx.x; i < 2 * num_acc; i += NT) sacc[i] = 0;
  // strip with HALF replicated samples around it (clamped reads = the reference's border extension): whole 16-byte chunks where
  // the chunk lies inside the picture, sample by sample at its borders
#pragma unroll
  for (int it = 0; it < (TR * CH + NT - 1) / NT; it++) {
    const int i = threadIdx.x + it * NT;
    if (i < TR * CH) {
      const int ty = i / CH, cx = i - ty * CH;
      const int y = min(max(y0 + ty - HALF, 0), h - 1), xs = x0 - 8 + 8 * cx;
      const int16_t* row = rec + (size_t)(y - r0) * pitch;
      uint4 v;
      if (xs >= 0 && xs + 8 <= w) v = __ldg(reinterpret_cast<const uint4*>(row + xs));
      else {
        uint32_t q[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const uint32_t a = (uint16_t)row[min(max(xs + 2 * j, 0), w - 1)], b = (uint16_t)row[min(max(xs + 2 * j + 1, 0), w - 1)];
          q[j] = a | (b << 16);
        }
        v = make_uint4(q[0], q[1], q[2], q[3]);
      }
      *reinterpret_cast<uint4*>(tile + ty * TP + 8 * cx) = v;
    }
  }
#pragma unroll
  for (int it = 0; it < (ST_H * (ST_W / 8)) / NT; it++) {
    const int i = threadIdx.x + it * NT;
    const int ty = i / (ST_W / 8), cx = i - ty * (ST_W / 8);
    if (y0 + ty < yend && x0 + 8 * cx < w)   // rows are padded to 64 samples: a chunk that starts inside the picture is readable
      *reinterpret_cast<uint4*>(sorg + ty * ST_W + 8 * cx) = __ldg(reinterpret_cast<const uint4*>(org + (size_t)(y0 + ty - r0) * pitch + x0 + 8 * cx));
  }
  __syncthreads();
  const int bj = threadIdx.x % (ST_W / 4), bi = threadIdx.x / (ST_W / 4);
  const int bx = x0 + 4 * bj, by = y0 + 4 * bi;
  const bool valid = bx < w && by < yend;
  int cls = 0;
  if (CLASSES && valid) cls = sd.alf_class[(size_t)((by - r0) >> 2) * g.units_w + (bx >> 2)];
  const int t = cls >> 5;
  // the block's transposed frame: sample (u, v) sits at P0 + u ex + v ey; transposeIdx 0: ex = (1, 0), ey = (0, 1); 1: (0, 1), (1, 0);
  // 2: (-1, 0), (0, 1) from the block's right edge; 3: (0, -1), (1, 0) from its bottom edge (EncAdaptiveLoopFilter.cpp:1463-1510)
  const int exx = t == 0 ? 1 : (t == 2 ? -1 : 0), exy = t == 1 ? 1 : (t == 3 ? -1 : 0);
  const int eyx = (t & 1) ? 1 : 0, eyy = (t & 1) ? 0 : 1;
  const int px0 = 4 * bj + (t == 2 ? 3 : 0), py0 = 4 * bi + (t == 3 ? 3 : 0);   // block-relative origin inside the strip
  const int sx = exx + exy * TP, sy = eyx + eyy * TP;
  const int c00 = (py0 + HALF) * TP + px0 + 8;
  int off[N - 1];
#pragma unroll
  for (int k = 0; k < N - 1; k++) { int a = 0, b = 0; tap_ab<HALF>(k, a, b); off[k] = a * sx + b * sy; }
  const int16_t* org0 = sorg + py0 * ST_W + px0;
  const int osx = exx + exy * ST_W, osy = eyx + eyy * ST_W;

  int acc[WORDS];
#pragma unroll
  for (int i = 0; i < WORDS; i++) acc[i] = 0;
#pragma unroll 1
  for (int s = 0; s < (valid ? 16 : 0); s++) {
    const int u = s & 3, v = s >> 2;
    const int c = c00 + u * sx + v * sy;
    int e[N];
#pragma unroll
    for (int k = 0; k < N - 1; k++) e[k] = tile[c + off[k]] + tile[c - off[k]];
    e[N - 1] = tile[c];
    const int yl = org0[u * osx + v * osy] - e[N - 1];
    int i = 0;
#pragma unroll
    for (int k = 0; k < N; k++)
#pragma unroll
      for (int l = k; l < N; l++) acc[i++] += e[k] * e[l];
#pragma unroll
    for (int k = 0; k < N; k++) acc[i++] += e[k] * yl;
    acc[i] += yl * yl;
  }
  // ---- (1) + (2): groups of lanes with the same (CTU, class) -> shared accumulators ----
  const int lane = threadIdx.x & 31;
  const int set = ((bx >> ctu_log2) - (x0 >> ctu_log2)) + sets_x * ((by >> ctu_log2) - (y0 >> ctu_log2));
  const int key = valid ? (CLASSES ? set * 25 + (cls & 31) : set) : 0x7FFF;
  // A warp whose 32 blocks share one (CTU, class) -- the usual case away from texture -- adds them with REDUX and goes to shared
  // memory once per word; in a mixed warp every lane adds its own sums (REDUX per group would run once per group, ~1000
  // instructions each), and lanes of the same class serialise on a word only among themselves.
  const bool uniform = __match_any_sync(0xFFFFFFFFu, key) == 0xFFFFFFFFu;
  uint32_t* lo = sacc + (valid ? key : 0) * WORDS;
  uint32_t* hi = lo + num_acc;
  auto add64 = [&](int i, long long v) {
    const uint32_t vl = (uint32_t)v;
    const uint32_t old = atomicAdd(lo + i, vl);
    const int vh = (int)(v >> 32) + ((uint32_t)(old + vl) < old ? 1 : 0);
    if (vh) atomicAdd(hi + i, (uint32_t)vh);
  };
  if (uniform) {
    if (valid) {   // (all 32 lanes are valid or none is: they share the key)
#pragma unroll
      for (int i = 0; i < WORDS; i++) {
        const unsigned sum_lo = __reduce_add_sync(0xFFFFFFFFu, (unsigned)acc[i] & 0xFFFFu);
        const int sum_hi = __reduce_add_sync(0xFFFFFFFFu, acc[i] >> 16);
        if (lane == (i & 31)) add64(i, ((long long)sum_hi << 16) + (long long)sum_lo);
      }
    }
  } else if (valid) {
#pragma unroll
    for (int i = 0; i < WORDS; i++) add64(i, (long long)acc[i]);
  }
  __syncthreads();
  // ---- (3): non-zero accumulators -> the CTUs' records ----
  for (int e = threadIdx.x; e < num_acc; e += NT) {
    const uint32_t l = sacc[e], hgh = sacc[num_acc + e];
    if (!(l | hgh)) continue;
    const int k = e / WORDS, i = e - k * WORDS;
    const int st = CLASSES ? k / 25 : k, c = CLASSES ? k - st * 25 : 0;
    // record row among the own CTU rows: the own rows start on a CTU row, so it follows from the tile row alone
    const int cx = (x0 >> ctu_log2) + st % sets_x, cy = (int)((blockIdx.y * ST_H) >> ctu_log2) + st / sets_x;
    long long* out = sd.alf_stats + (size_t)(cy * g.ctus_w + cx) * ILF_ALF_STATS_WORDS + (plane == 0 ? (size_t)c * WORDS : (size_t)(25 * 105 + (plane - 1) * 36)) + i;
    atomicAdd(reinterpret_cast<unsigned long long*>(out), ((unsigned long long)hgh << 32) | l);
  }
}

}  // namespace

// The slots' class maps (SlotDev::alf_class) must be current: launch_alf_classify first.  The records must be zero.
void launch_alf_stats(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st) {
  auto sets = [&](int sh) { const int l = g.ctu_log2 - sh; return std::max(1, ST_W >> l) * std::max(1, ST_H >> l); };
  const int smem_y = sets(0) * 25 * Shape<3>::WORDS * 8, smem_c = sets(1) * Shape<2>::WORDS * 8;
  if (smem_y > 36 * 1024) cudaFuncSetAttribute(alf_stats_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_y);   // CTUs below 128: several records per tile
  alf_stats_kernel<3, true><<<dim3((g.width + ST_W - 1) / ST_W, (g.out_rows + ST_H - 1) / ST_H, num_slots), NT, smem_y, st>>>(g, slots, first_slot, ctl, 0);
  const dim3 gc((g.width / 2 + ST_W - 1) / ST_W, (g.out_rows / 2 + ST_H - 1) / ST_H, num_slots);
  alf_stats_kernel<2, false><<<gc, NT, smem_c, st>>>(g, slots, first_slot, ctl, 1);
  alf_stats_kernel<2, false><<<gc, NT, smem_c, st>>>(g, slots, first_slot, ctl, 2);
}

}  // namespace ilf
