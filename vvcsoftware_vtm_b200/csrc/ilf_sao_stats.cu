// ilf_sao_stats.cu -- encoder-side SAO statistics (SURVEY.md 8f rank 2) on the device-resident deblocked picture (sm_100a).
//
// Replaces EncSampleAdaptiveOffset::getStatistics (EncoderLib/EncSampleAdaptiveOffset.cpp:278-331) and its per-block worker
// getBlkStats (:1122-1487) for the path the encoder takes without SaoCtuBoundary: for every CTU, component and SAO type
// (EO 0/90/135/45 degrees, BO) the number of samples per class and the sum of (original - deblocked) per class.  The
// samples of a CTU block that contribute depend on the type, on the neighbour-CTU availability and on the skip lines of
// createEncData (:122-128): the last 5 (chroma 3) columns and 4 (2) rows of a CTU are left out when the right / below CTU
// exists; the first row of the two diagonal types has its own column range (:1278-1287, :1360-1372).
//
// One CTA per (CTU, component).  A warp owns a strip of 32 columns and walks it downwards with a rolling 3x3 window in
// registers (three loads per sample row: the row below, L1 resident for the two neighbours); the eight signs of a sample give
// its four edge classes.  Accumulation needs no atomics and no class-indexed registers: every (warp, type, class) has 32
// words of shared memory, one per lane, and a sample adds (diff << 8) + 1 to the word of its class -- count (at most 128 per
// lane and CTU) and sum of differences travel in one 32-bit word (20 + 8 bits), bank = lane, so the read-modify-write is
// conflict-free.  At the end every warp reduces its words (REDUX), one shared-memory atomic per class and warp builds the
// CTA totals, and the CTA writes the 5 x 64 int64 words of SAOStatData.
// Bound: HBM reads of two pictures (6 B per luma pixel); the output is 7.7 KB per CTU.
// A band context measures its own CTUs (record = blockIdx.x): decisions in picture coordinates, plane rows addressed from the first
// held row.  Its rows reach one deblocked row beyond the own rows, inside the 16-row halo.
#include "ilf_common.cuh"

namespace ilf {
namespace {

#ifndef SAO_STATS_THREADS
#define SAO_STATS_THREADS 128
#endif
constexpr int NT = SAO_STATS_THREADS, NW = NT / 32;
constexpr int CNT_BITS = 8;   // a lane sees at most 128 rows of a CTU: count < 2^8, |sum of differences| < 2^19 (12 bit) -> one 32-bit word
constexpr int EO_WORDS = 4 * 5 * 32, BO_WORDS = 32 * 32, WARP_WORDS = EO_WORDS + BO_WORDS;  // per warp: [type][class][lane], [band][lane]
constexpr int SMEM_BYTES = NW * WARP_WORDS * 4;

__device__ __forceinline__ int sgn3(int a, int b) { return min(max(a - b, -1), 1); }

__global__ void __launch_bounds__(NT, 1024 / NT) sao_stats_kernel(Geom g, const SlotDev* __restrict__ slots, int first_slot, BatchCtl bc) {
  extern __shared__ __align__(16) int acc_all[];
  __shared__ int tot[5][64];
  pdl_launch_dependents();
  const SlotDev& sd = slots[first_slot + bc.slot[blockIdx.z]];
  const unsigned ctl = bc.v[blockIdx.z];
  const int comp = blockIdx.y, ctu = blockIdx.x + (g.out_row0 >> g.ctu_log2) * g.ctus_w, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cx = ctu % g.ctus_w, cy = ctu / g.ctus_w;
  const int sh = comp ? 1 : 0, csz = 1 << g.ctu_log2;
  const int lx0 = cx << g.ctu_log2, ly0 = cy << g.ctu_log2;
  const int pw = g.width >> sh, ph = g.height >> sh, pitch = comp ? g.pitch_c : g.pitch_y;
  const int x0 = lx0 >> sh, y0 = ly0 >> sh;
  const int w = min(csz, g.width - lx0) >> sh, h = min(csz, g.height - ly0) >> sh;
  const unsigned av = sd.stats_avail[ctu];
  const bool L = av & ILF_AVAIL_L, A = av & ILF_AVAIL_A, AL = av & ILF_AVAIL_AL;
  const bool R = lx0 + csz < g.width, B = ly0 + csz < g.height, AR = ly0 > 0 && R;
  const int skip_r = comp ? 3 : 5, skip_b = comp ? 2 : 4;
  // column / row ranges per type (getBlkStats, isCalculatePreDeblockSamples == false)
  const int sx_e = L ? 0 : 1, ex_e = R ? w - skip_r : w - 1;       // EO 0 / 135 / 45 columns
  const int ey_0 = B ? h - skip_b : h;                              // EO 0 and BO rows
  const int ex_90 = R ? w - skip_r : w, sy_90 = A ? 0 : 1, ey_d = B ? h - skip_b : h - 1;  // EO 90 columns; rows of 90 / 135 / 45
  const int fs_135 = AL ? 0 : 1, fe_135 = A ? ex_e : 1;             // first row of EO 135
  const int fs_45 = A ? sx_e : ex_e, fe_45 = (!R && AR) ? w : ex_e;  // first row of EO 45
  const int bo_shift = (comp ? g.bd_chroma : g.bd_luma) - 5;

  int* acc = acc_all + warp * WARP_WORDS;
  for (int i = lane; i < WARP_WORDS; i += 32) acc[i] = 0;
  for (int i = tid; i < 5 * 64; i += NT) (&tot[0][0])[i] = 0;
  __syncthreads();
  pdl_wait();  // the deblocking kernel has written the picture read from here on

  // strips of 32 columns x row groups (NW warps): 128-wide luma = 4 strips x 1 row group, 64-wide chroma = 2 x 2
  const int nstrips = (w + 31) >> 5, nrg = NW / nstrips;
  const int strip = warp % nstrips, rg = warp / nstrips;
  const int rh = (h + nrg - 1) / nrg;
  const int ya = rg * rh, yb = min(h, ya + rh);
  const int x = 32 * strip + lane;
  if (rg < nrg && ya < yb) {
    const int16_t* __restrict__ src = sd.buf[ctl_src(ctl, comp)][comp];
    const int16_t* __restrict__ org = sd.org[comp];
    const int gx = min(x0 + x, pw - 1), gxl = max(gx - 1, 0), gxr = min(gx + 1, pw - 1);
    const bool xin = x < w;
    const bool x_e = xin && x >= sx_e && x < ex_e, x_90 = xin && x < ex_90, x_135f = xin && x >= fs_135 && x < fe_135, x_45f = xin && x >= fs_45 && x < fe_45;
    int* bo = acc + EO_WORDS + lane;    // + band * 32
    // 32-bit sample indices (a plane has < 2^31 samples)
    const int oL = gxl - gx, oR = gxr - gx;
    const int col = gx - (g.row0 >> sh) * pitch;   // sample index of picture row 0 in this column (held rows start at row0)
    int iu = max(y0 + ya - 1, 0) * pitch + col, ic = (y0 + ya) * pitch + col;
    int ul = src[iu + oL], u = src[iu], ur = src[iu + oR];
    int l = src[ic + oL], c = src[ic], r = src[ic + oR];
    const int e0 = 2 * 32 * 4, e1 = e0 + 160 * 4, e2 = e0 + 320 * 4, e3 = e0 + 480 * 4;  // byte offsets of class 0 of every EO type
    char* accb = reinterpret_cast<char*>(acc + lane);
    char* bob = reinterpret_cast<char*>(bo);
    // Rows go four at a time: the sixteen loads of a group are issued before the first of them is used, so a warp keeps
    // 1 KB in flight (32 resident warps per SM: 32 KB) instead of the 128 bytes of one row.
    constexpr int G = 4;
    for (int yg = ya; yg < yb; yg += G) {
      int D[G][3], O[G];
#pragma unroll
      for (int k = 0; k < G; k++) {
        const int gy = y0 + yg + k;
        const int id = min(gy + 1, ph - 1) * pitch + col;
        D[k][0] = src[id + oL]; D[k][1] = src[id]; D[k][2] = src[id + oR];
        O[k] = org[min(gy, ph - 1) * pitch + col];
      }
#pragma unroll
      for (int k = 0; k < G; k++) {
        const int y = yg + k;
        if (y < yb) {
          const int dl = D[k][0], d = D[k][1], dr = D[k][2];
          const int v = ((O[k] - c) << CNT_BITS) + 1;   // (diff << 8) + count
          const int c0 = sgn3(c, l) + sgn3(c, r), c1 = sgn3(c, u) + sgn3(c, d), c2 = sgn3(c, ul) + sgn3(c, dr), c3 = sgn3(c, ur) + sgn3(c, dl);
          const bool first = y == 0, yd = y < ey_d, y0r = y < ey_0;
          // the five words are distinct (different types): all loads first, then the stores
          int* p0 = reinterpret_cast<int*>(accb + e0 + c0 * 128);
          int* p1 = reinterpret_cast<int*>(accb + e1 + c1 * 128);
          int* p2 = reinterpret_cast<int*>(accb + e2 + c2 * 128);
          int* p3 = reinterpret_cast<int*>(accb + e3 + c3 * 128);
          int* pb = reinterpret_cast<int*>(bob + (c >> bo_shift) * 128);
          const int a0 = *p0, a1 = *p1, a2 = *p2, a3 = *p3, ab = *pb;
          if (y0r && x_e) *p0 = a0 + v;
          if (y >= sy_90 && yd && x_90) *p1 = a1 + v;
          if (yd && (first ? x_135f : x_e)) *p2 = a2 + v;
          if (yd && (first ? x_45f : x_e)) *p3 = a3 + v;
          if (y0r && x_90) *pb = ab + v;   // BO: the columns of EO 90, the rows of EO 0
          ul = l; u = c; ur = r; l = dl; c = d; r = dr;
        }
      }
    }
  }
  __syncwarp();
  // Every warp folds its lanes.  Lane j sums the 32 words of row j (skewed, so that the lanes hit different banks):
  // word = diff * 256 + count with count < 256.
  for (int base = 0; base < 20 + 32; base += 32) {
    const int rowi = base + lane;
    if (rowi < 20 + 32) {
      int sd = 0, sn = 0;
#pragma unroll 8
      for (int k = 0; k < 32; k++) {
        const int wd = acc[rowi * 32 + ((k + lane) & 31)];
        const int n = wd & ((1 << CNT_BITS) - 1);
        sn += n; sd += (wd - n) >> CNT_BITS;
      }
      if (sn) {
        const int t = rowi < 20 ? rowi / 5 : 4, k = rowi < 20 ? rowi % 5 : rowi - 20;
        atomicAdd(&tot[t][32 + k], sn);
        atomicAdd(&tot[t][k], sd);
      }
    }
  }
  __syncthreads();
  // SAOStatData layout: [type][diff[32], count[32]] int64
  long long* out = sd.stats + ((size_t)blockIdx.x * 3 + comp) * (5 * 64);
  for (int i = tid; i < 5 * 64; i += NT) out[i] = (&tot[0][0])[i];
}

}  // namespace

void launch_sao_stats(const Geom& g, const SlotDev* slots, int first_slot, int num_slots, const BatchCtl& ctl, cudaStream_t st) {
  static bool attr_set[64] = {};
  once_per_device(attr_set, [&] { cudaFuncSetAttribute(sao_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES); });
  const int ctu_rows = ((g.out_row0 + g.out_rows - 1) >> g.ctu_log2) - (g.out_row0 >> g.ctu_log2) + 1;   // own CTU rows
  launch_pdl(sao_stats_kernel, dim3(g.ctus_w * ctu_rows, 3, num_slots), dim3(NT), SMEM_BYTES, st, g, slots, first_slot, ctl);
}

}  // namespace ilf
