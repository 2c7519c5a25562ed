// ilf_hash.cu -- decoded-picture hash of the device-resident picture: CRC and checksum (sm_100a).
//
// Replaces calcCRC / calcChecksum (source/Lib/CommonLib/PicYuvMD5.cpp:91-175), the two SEI hash methods that are not inherently
// serial (MD5 is, and stays on the host): the decoder compares them with the decoded-picture-hash SEI after the in-loop filters
// (DecLib.cpp:579-588), so a hash taken where the filtered picture already is needs 12 bytes of device -> host traffic instead
// of waiting for the 25 MB picture.
//
// CRC (compCRC): a 16-bit register, message bits shifted in at the bottom, polynomial 0x1021 fed back from the top -- linear over
// GF(2): after n bits  s_n = M^n s_0 + R(bits).  Every thread walks ONE row from a zero register (bytewise with a 256-entry table,
// low byte then high byte of each sample); rows are equally long, so a row advances the register by the same matrix
// A = M^(bits per row), and a tree over the rows (front-padded with empty rows to a power of two, level l combining with
// A^(2^l)) gives R(picture) from a zero register.  The host finishes: the 0xffff start value and the 16 appended zero bits are
// two more matrix products.  Checksum (compChecksum): a plain sum of masked bytes, reduced next to the CRC.
//
// The kernels hash a window of rows: the whole picture, or the own rows of a band context (the row origin of the window keeps the
// checksum's row mask in picture coordinates).  Parts of consecutive rows combine on the host (ilf_hash_combine): a part of n rows
// advances the register by A^n, so folding s = A^n s + R(part) over the parts in row order gives R(picture).
#include <algorithm>
#include <vector>

#include "ilf_common.cuh"

namespace ilf {
namespace {

__constant__ uint16_t c_crc_tab[256];            // register (v << 8) after 8 zero bits

__device__ __forceinline__ uint32_t crc_byte(const uint16_t* tab, uint32_t s, uint32_t b) { return (((s << 8) | b) & 0xffffu) ^ tab[s >> 8]; }
__device__ __forceinline__ uint32_t mat_apply(const uint16_t* col, uint32_t s) {
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) r ^= (s >> i) & 1 ? col[i] : 0;
  return r;
}

struct HashArgs {
  const int16_t* plane[3];
  int pitch[3], width[3], height[3], bd[3], padded[3];  // height = rows of the window; padded = rows rounded up to a power of two
  int y0[3];                                             // picture row of the window's first row (checksum mask)
  uint32_t* rows;                                        // [3][16384] {crc | checksum hi?} -> two arrays
  uint32_t* sums;
  uint16_t pow[3][14][16];                               // per plane: columns of A^(2^l), A = one row's worth of register steps
};

// one thread per row: zero-register CRC and checksum of the row
__global__ void __launch_bounds__(32) hash_rows_kernel(HashArgs a) {
  __shared__ uint16_t tab[256];   // the lanes index it with different values: shared memory, not the constant cache
  for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = c_crc_tab[i];
  __syncthreads();
  const int p = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.height[p]) return;
  const int w = a.width[p];
  const bool two = a.bd[p] > 8;
  const uint4* row = reinterpret_cast<const uint4*>(a.plane[p] + (size_t)r * a.pitch[p]);
  uint32_t s = 0, sum = 0;
  const int y = a.y0[p] + r;
  const uint32_t my = (y & 0xff) ^ (y >> 8);
  auto sample = [&](uint32_t smp, int x) {
    const uint32_t mask = (my ^ (x & 0xff) ^ (x >> 8)) & 0xff;
    s = crc_byte(tab, s, smp & 0xff);
    sum += (smp & 0xff) ^ mask;
    if (two) { s = crc_byte(tab, s, smp >> 8); sum += (smp >> 8) ^ mask; }
  };
  for (int x8 = 0; x8 < w / 8; x8++) {
    const uint4 v = __ldg(row + x8);
    const uint32_t wds[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 8; k++) sample((wds[k >> 1] >> (16 * (k & 1))) & 0xffffu, 8 * x8 + k);
  }
  for (int x = w & ~7; x < w; x++) sample((uint16_t)a.plane[p][(size_t)r * a.pitch[p] + x], x);   // chroma widths are multiples of 4 only
  a.rows[p * 16384 + (a.padded[p] - a.height[p]) + r] = s;
  a.sums[p * 16384 + r] = sum;
}

// one block per plane: tree over the (front-padded) rows
__global__ void __launch_bounds__(1024) hash_reduce_kernel(HashArgs a, uint32_t* out /* [3][2] */) {
  __shared__ uint32_t sh[16384 / 2];
  __shared__ uint32_t ssum[32];
  const int p = blockIdx.x, n = a.padded[p], pad = n - a.height[p], tid = threadIdx.x;
  const uint32_t* rows = a.rows + p * 16384;
  // level 0 straight from global memory
  for (int i = tid; i < n / 2; i += 1024) {
    const uint32_t l = 2 * i >= pad ? rows[2 * i] : 0, r = 2 * i + 1 >= pad ? rows[2 * i + 1] : 0;
    sh[i] = n >= 2 ? mat_apply(a.pow[p][0], l) ^ r : 0;
  }
  __syncthreads();
  int lvl = 1;
  for (int m = n / 4; m >= 1; m >>= 1, lvl++) {
    uint32_t v[4];
    int cnt = 0;
    for (int i = tid; i < m; i += 1024) v[cnt++] = mat_apply(a.pow[p][lvl], sh[2 * i]) ^ sh[2 * i + 1];
    __syncthreads();
    cnt = 0;
    for (int i = tid; i < m; i += 1024) sh[i] = v[cnt++];
    __syncthreads();
  }
  uint32_t sum = 0;
  for (int i = tid; i < a.height[p]; i += 1024) sum += a.sums[p * 16384 + i];
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((tid & 31) == 0) ssum[tid >> 5] = sum;
  __syncthreads();
  if (tid == 0) {
    uint32_t t = 0;
    for (int i = 0; i < 32; i++) t += ssum[i];
    out[2 * p] = n >= 2 ? sh[0] : rows[0];
    out[2 * p + 1] = t;
  }
}

// ---- GF(2) helpers on the host: 16x16 matrices as 16 columns ----
struct Mat { uint16_t col[16]; };
uint16_t step(uint16_t s) { return (uint16_t)(((s << 1) & 0xffff) ^ ((s >> 15) ? 0x1021 : 0)); }
uint16_t apply(const Mat& m, uint16_t s) { uint16_t r = 0; for (int i = 0; i < 16; i++) if ((s >> i) & 1) r ^= m.col[i]; return r; }
Mat mul(const Mat& a, const Mat& b) { Mat r; for (int i = 0; i < 16; i++) r.col[i] = apply(a, b.col[i]); return r; }
Mat mat_pow_bits(unsigned long long nbits) {  // M^nbits
  Mat base, res;
  for (int i = 0; i < 16; i++) { base.col[i] = step((uint16_t)(1u << i)); res.col[i] = (uint16_t)(1u << i); }
  while (nbits) { if (nbits & 1) res = mul(base, res); base = mul(base, base); nbits >>= 1; }
  return res;
}

}  // namespace

// planes[p]: device pointers of the held planes.  reg / sum: R(rows) from a zero register and the checksum partial sum of luma rows
// [first, first + n) of the held planes (chroma rows halved); y0 = picture row of `first`.
cudaError_t hash_rows(const Geom& g, const int16_t* const planes[3], uint32_t* scratch /* 2 * 3 * 16384 + 8 words */, cudaStream_t st, int first, int n, int y0,
                      uint32_t reg[3], uint32_t sum[3]) {
  static bool tab_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  HashArgs a;
  for (int p = 0; p < 3; p++) {
    const int sh = p ? 1 : 0;
    a.pitch[p] = p ? g.pitch_c : g.pitch_y;
    a.plane[p] = planes[p] + (size_t)(first >> sh) * a.pitch[p];
    a.width[p] = g.width >> sh;
    a.height[p] = n >> sh;
    a.y0[p] = y0 >> sh;
    a.bd[p] = p ? g.bd_chroma : g.bd_luma;
    int m = 1;
    while (m < a.height[p]) m <<= 1;
    a.padded[p] = m;
    Mat mp = mat_pow_bits((unsigned long long)a.width[p] * (a.bd[p] > 8 ? 16 : 8));
    for (int l = 0; l < 14; l++) { for (int i = 0; i < 16; i++) a.pow[p][l][i] = mp.col[i]; mp = mul(mp, mp); }
  }
  a.rows = scratch;
  a.sums = scratch + 3 * 16384;
  uint32_t* out = scratch + 6 * 16384;
  if (dev >= 0 && dev < 64 && !tab_set[dev]) {
    uint16_t tab[256];
    for (int v = 0; v < 256; v++) { uint16_t s = (uint16_t)(v << 8); for (int b = 0; b < 8; b++) s = step(s); tab[v] = s; }
    cudaMemcpyToSymbolAsync(c_crc_tab, tab, sizeof(tab), 0, cudaMemcpyHostToDevice, st);
    tab_set[dev] = true;
  }
  const int maxh = a.height[0];
  hash_rows_kernel<<<dim3((maxh + 31) / 32, 3), 32, 0, st>>>(a);   // one warp per CTA: the 4320 row walks of a 4K picture spread over all SMs
  hash_reduce_kernel<<<3, 1024, 0, st>>>(a, out);
  uint32_t h[6];
  cudaError_t e = cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, st);
  if (e != cudaSuccess) return e;
  e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return e;
  for (int p = 0; p < 3; p++) {
    reg[p] = h[2 * p];
    sum[p] = h[2 * p + 1];
  }
  return cudaGetLastError();
}

// The register compCRC leaves after `bits` message bits from 0xffff whose contribution from a zero register is `reg`, followed by
// the 16 appended zero bits.
static uint32_t crc_finish(uint16_t reg, unsigned long long bits) {
  const uint16_t s = (uint16_t)(apply(mat_pow_bits(bits), 0xffff) ^ reg);
  return apply(mat_pow_bits(16), s);
}

cudaError_t picture_hash(const Geom& g, const int16_t* const planes[3], uint32_t* scratch, cudaStream_t st, uint32_t out_crc[3], uint32_t out_sum[3]) {
  uint32_t reg[3];
  cudaError_t e = hash_rows(g, planes, scratch, st, 0, g.height, 0, reg, out_sum);
  if (e != cudaSuccess) return e;
  for (int p = 0; p < 3; p++) {
    const unsigned long long row_bits = (unsigned long long)(g.width >> (p ? 1 : 0)) * ((p ? g.bd_chroma : g.bd_luma) > 8 ? 16 : 8);
    out_crc[p] = crc_finish((uint16_t)reg[p], row_bits * (unsigned long long)(g.height >> (p ? 1 : 0)));
  }
  return cudaSuccess;
}

}  // namespace ilf

// Host only: parts may come from other processes, so everything is checked before it is used.
extern "C" int ilf_hash_combine(const ilf_hash_part* parts, int num_parts, int kind, uint32_t out[3]) {
  using namespace ilf;
  if (!parts || !out || num_parts < 1 || (kind != ILF_HASH_CRC && kind != ILF_HASH_CHECKSUM)) return ILF_ERR_ARG;
  const ilf_hash_part& p0 = parts[0];
  if (p0.width <= 0 || p0.height <= 0 || ((p0.width | p0.height) & 1) || p0.bd_luma < 8 || p0.bd_luma > 12 || p0.bd_chroma < 8 || p0.bd_chroma > 12) return ILF_ERR_ARG;
  std::vector<const ilf_hash_part*> order(num_parts);
  for (int i = 0; i < num_parts; i++) {
    const ilf_hash_part& q = parts[i];
    if (q.width != p0.width || q.height != p0.height || q.bd_luma != p0.bd_luma || q.bd_chroma != p0.bd_chroma) return ILF_ERR_ARG;
    if (q.first_row < 0 || q.num_rows < 1 || (long long)q.first_row + q.num_rows > p0.height) return ILF_ERR_ARG;
    if ((q.first_row | q.num_rows) & 1) return ILF_ERR_ARG;   // even rows: chroma rows are exactly half
    order[i] = &q;
  }
  std::sort(order.begin(), order.end(), [](const ilf_hash_part* a, const ilf_hash_part* b) { return a->first_row < b->first_row; });
  long long next = 0;   // the parts tile [0, height): no gap, no overlap (each part lies inside the picture, so no overflow)
  for (const ilf_hash_part* q : order) {
    if (q->first_row != next) return ILF_ERR_ARG;
    next += q->num_rows;
  }
  if (next != p0.height) return ILF_ERR_ARG;
  for (int p = 0; p < 3; p++) {
    const int sh = p ? 1 : 0;
    const unsigned long long row_bits = (unsigned long long)(p0.width >> sh) * ((p ? p0.bd_chroma : p0.bd_luma) > 8 ? 16 : 8);
    uint16_t s = 0;
    uint32_t sum = 0;
    for (const ilf_hash_part* q : order) {
      s = (uint16_t)(apply(mat_pow_bits(row_bits * (unsigned long long)(q->num_rows >> sh)), s) ^ (uint16_t)q->crc[p]);
      sum += q->sum[p];
    }
    out[p] = kind == ILF_HASH_CRC ? crc_finish(s, row_bits * (unsigned long long)(p0.height >> sh)) : sum;
  }
  return ILF_OK;
}
