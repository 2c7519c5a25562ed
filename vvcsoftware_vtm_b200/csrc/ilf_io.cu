// ilf_io.cu -- pictures to and from device memory of the caller (ilf_upload_device, ilf_set_original_device, ilf_download_device):
// one kernel copies the three planes between the caller's pitched planes and the slot's, converting the sample type (int16 or
// uint8) and the bit depth on the way.
//
// Per plane a sample v (int16 containers read as unsigned 16-bit, uint8 as unsigned 8-bit) becomes, in int32,
//   v << up                                              when the destination is deeper (up = dst depth - src depth > 0)
//   clip3(0, maxv, (v + (1 << (down - 1))) >> down)      when it is shallower (down = src depth - dst depth > 0, maxv = 2^dst - 1)
//   v                                                    when the depths are equal
// and is stored as the destination type (the low 16 or 8 bits).  Every combination, the identity included, is the same kernel.
//
// A CTA of 128 threads copies one row of one plane (a 4K luma row is 240 groups of 16 samples, a chroma row 120).  Where the source
// and the destination rows can both be addressed in 16-byte words after the same head of samples, the row body moves in groups of
// 16 samples (one or two 16-byte loads, one or two 16-byte stores); the head, the tail and rows whose alignments never meet (for
// example a uint8 view with an odd pitch) move a sample at a time.  The kernel's name, ilf::ilf_io_convert, is what profiles show.
#include "ilf_common.cuh"

namespace ilf {

namespace {

__device__ __forceinline__ int io_convert(int v, const IoPlane& p) {
  return p.down ? clip3i(0, p.maxv, (v + (1 << (p.down - 1))) >> p.down) : v << p.up;
}

__device__ __forceinline__ int io_load1(const unsigned char* row, int x, int bytes) {
  return bytes == 2 ? (int)reinterpret_cast<const uint16_t*>(row)[x] : (int)row[x];
}

__device__ __forceinline__ void io_store1(unsigned char* row, int x, int bytes, int v) {
  if (bytes == 2) reinterpret_cast<uint16_t*>(row)[x] = (uint16_t)v;
  else row[x] = (unsigned char)v;
}

// 16 samples from a 16-byte aligned address: two words of int16 or one of uint8.
__device__ __forceinline__ void io_load16(const unsigned char* p, int bytes, int v[16]) {
  if (bytes == 2) {
    const uint4 a = ldg_u4(p), b = ldg_u4(p + 16);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; i++) { v[2 * i] = (int)(w[i] & 0xFFFFu); v[2 * i + 1] = (int)(w[i] >> 16); }
  } else {
    const uint4 a = ldg_u4(p);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) v[4 * i + j] = (int)((w[i] >> (8 * j)) & 0xFFu);
  }
}

__device__ __forceinline__ void io_store16(unsigned char* p, int bytes, const int v[16]) {
  if (bytes == 2) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = ((uint32_t)v[2 * i] & 0xFFFFu) | ((uint32_t)v[2 * i + 1] << 16);
    reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
    reinterpret_cast<uint4*>(p)[1] = make_uint4(w[4], w[5], w[6], w[7]);
  } else {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; i++)
      w[i] = ((uint32_t)v[4 * i] & 0xFFu) | ((uint32_t)v[4 * i + 1] & 0xFFu) << 8 | ((uint32_t)v[4 * i + 2] & 0xFFu) << 16 | (uint32_t)v[4 * i + 3] << 24;
    reinterpret_cast<uint4*>(p)[0] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

}  // namespace

// blockIdx.x = row over the three planes: rows [0, p[0].h) of plane 0, then those of plane 1 and plane 2.
__global__ void __launch_bounds__(128) ilf_io_convert(IoBatch b) {
  int r = blockIdx.x, pi = 0;
  while (pi < 2 && r >= b.p[pi].h) { r -= b.p[pi].h; pi++; }
  const IoPlane& p = b.p[pi];
  const int sb = b.src_bytes, db = b.dst_bytes, w = p.w;
  const unsigned char* src = static_cast<const unsigned char*>(p.src) + (long long)r * p.src_pitch;
  unsigned char* dst = static_cast<unsigned char*>(p.dst) + (long long)r * p.dst_pitch;
  // head: samples until the destination is 16-byte aligned; the body runs when the source is aligned there as well
  int head = (int)(((16 - ((uintptr_t)dst & 15)) & 15) / db);
  if (head > w) head = w;
  const bool vec = (((uintptr_t)src + (size_t)head * sb) & 15) == 0;
  const int groups = vec ? (w - head) >> 4 : 0;
  if (!vec) head = w;   // the whole row a sample at a time
  const int body_end = head + 16 * groups, scalar = head + (w - body_end);
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    int v[16];
    io_load16(src + (size_t)(head + 16 * g) * sb, sb, v);
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = io_convert(v[i], p);
    io_store16(dst + (size_t)(head + 16 * g) * db, db, v);
  }
  for (int k = threadIdx.x; k < scalar; k += blockDim.x) {
    const int x = k < head ? k : body_end + (k - head);
    io_store1(dst, x, db, io_convert(io_load1(src, x, sb), p));
  }
}

void launch_io_convert(const IoBatch& b, cudaStream_t st) {
  const int rows = b.p[0].h + b.p[1].h + b.p[2].h;
  if (rows > 0) ilf_io_convert<<<rows, 128, 0, st>>>(b);
}

}  // namespace ilf
