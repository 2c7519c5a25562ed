// ilf_api.cu -- the extern "C" boundary of libilf_b200.so (see include/ilf_b200.h): contexts, device-resident
// planes, pinned async transfers, side-information upload and stage launches.  No CPU fallback anywhere.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <unistd.h>

#include "ilf_common.cuh"
#include "ilf_alf_tab.cuh"

using namespace ilf;

namespace {

thread_local std::string g_create_error;

constexpr int ALF_DP_WORDS = 25 * 4 * alftab::LUMA_WORDS + alftab::CHROMA_WORDS;

// Pageable host planes (the reference's PelStorage) go through page-locked staging buffers.  A single memcpy thread moves about
// 8 GB/s, a 4K picture is 25 MB each way, so the staging copies are cut into row chunks that a few helper threads copy while the
// DMA engine already moves the chunks that are done (upload), or as soon as the DMA engine has delivered them (download).
// Page-locking the caller's planes instead (cudaHostRegister) costs 20 - 300 ms per plane set on the boxes measured and goes stale
// when the owner frees or recycles the memory, so the library never does that on its own.  ILF_COPY_THREADS (default 4; 1 = inline).
class CopyPool {
 public:
  ~CopyPool() {
    { std::lock_guard<std::mutex> l(m_); stop_ = true; }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  int threads() {
    static const int n = getenv("ILF_COPY_THREADS") ? std::max(1, atoi(getenv("ILF_COPY_THREADS"))) : 4;
    return n;
  }
  // runs fn(0 .. ntasks-1) on the helper threads; returns at once.  One batch at a time (wait() before the next).
  void start(int ntasks, std::function<void(int)> fn) {
    if (th_.empty()) for (int i = 0; i < threads(); i++) th_.emplace_back([this] { loop(); });
    { std::lock_guard<std::mutex> l(m_); fn_ = std::move(fn); ntasks_ = ntasks; next_ = 0; done_ = 0; gen_++; }
    cv_.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> l(m_);
    cv_done_.wait(l, [this] { return done_ == ntasks_; });
  }
 private:
  void loop() {
    unsigned long long seen = 0;
    for (;;) {
      std::unique_lock<std::mutex> l(m_);
      cv_.wait(l, [&] { return stop_ || (gen_ != seen && next_ < ntasks_); });
      if (stop_) return;
      const unsigned long long g = gen_;
      while (gen_ == g && next_ < ntasks_) {
        const int i = next_++;
        l.unlock();
        fn_(i);
        l.lock();
        if (++done_ == ntasks_) cv_done_.notify_all();
      }
      seen = g;
    }
  }
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable cv_, cv_done_;
  std::function<void(int)> fn_;
  int ntasks_ = 0, next_ = 0, done_ = 0;
  unsigned long long gen_ = 0;
  bool stop_ = false;
};
constexpr int COPY_CHUNKS_MAX = 24;
struct CopyChunk { int plane, row0, rows; size_t stage_off; };  // rows of one plane; offset into the staging buffer in samples

struct Slot {
  int16_t* planes = nullptr;   // one allocation: 3 buffers x (Y, Cb, Cr)
  uint32_t* info = nullptr;
  uint32_t* info_c = nullptr;
  void* mv = nullptr;          // int16x4 or int32x4 per unit
  void* db_rec = nullptr;      // deblocking edge records (db_rec_layout), derived by ilf_set_deblock_info
  uint8_t* ctu_slice = nullptr;
  ilf_deblock_params* db_params = nullptr;
  ilf_sao_ctu* sao = nullptr;
  ilf_alf_params* alf = nullptr;
  int* alf_coef = nullptr;     // [25][4][16] transposed luma coefficient table
  uint32_t* alf_coef_dp = nullptr;  // [25][4][20] + [16]: dot-product layout of the luma filters and of the chroma filter (ilf_alf_tab.cuh)
  uint8_t* alf_ctu_enable = nullptr;
  uint8_t* alf_class = nullptr;
  int16_t* org = nullptr;      // source picture of the encoder (3 planes, same layout as one buffer of `planes`); allocated by ilf_set_original
  uint8_t* stats_avail = nullptr;
  long long* stats = nullptr;  // [num_ctus][3][5][64]
  long long* alf_stats = nullptr;  // [num_ctus][ILF_ALF_STATS_WORDS]
  bool has_org = false;
  bool org_since_upload = false;   // ilf_set_original was called after the slot's last upload (ilf_deblock_search)
  int search_k = 0;                // candidates of the slot's last ilf_deblock_search (0: none yet)
  int16_t* pinned = nullptr;   // host staging for pageable planes on the way up, one picture; allocated on first use
  int16_t* pinned_down = nullptr;  // ... and on the way down
  uint8_t* pinned_side = nullptr;  // host staging for side information
  size_t pinned_side_bytes = 0;
  SlotDev dev;                 // host copy of the device descriptor
  SlotDev pushed;              // what the device copy holds (valid once pushed_valid): unchanged descriptors are not sent again
  bool pushed_valid = false;
  bool uploaded = false, has_db = false, has_sao = false, has_alf = false, has_ctree = false;
  int mv_mode = 0;             // 0 none, 1 int16, 2 int32
  int result_buf[3] = {0, 0, 0};  // buffer holding the current picture, per plane
  bool sao_on[3] = {false, false, false};  // any CTU with SAO enabled, per component
  bool alf_on[3] = {false, false, false};
  bool db_chroma = true;           // the chroma decisions' grid has an intra unit: deblocking may change the chroma planes
  bool alf_is7 = false;            // luma filter shape of the slot's ALF parameters
  // ordering of the slot's copies and kernels (see "Per-slot ordering" above join())
  cudaEvent_t ev_up = nullptr, ev_run = nullptr, ev_down = nullptr;
  cudaEvent_t ev_rec = nullptr;    // the slot's last deblocking record pass is done; rec_pending: issued since a stream last waited for it
  bool rec_pending = false;
  cudaStream_t run_stream = nullptr;
  cudaEvent_t ev_side[3] = {nullptr, nullptr, nullptr};
  size_t side_off[4] = {0, 0, 0, 0};                       // regions of pinned_side per stage
  bool h2d_pending = false, d2h_pending = false;
  // band mode: planes of the neighbouring bands' matching slot (above, below)
  struct Neighbour { const int16_t* planes = nullptr; void* ipc_base = nullptr; int device = -1, row0 = 0, rows = 0, pitch_y = 0, pitch_c = 0; size_t plane_y = 0, plane_c = 0; } nb[2];
};

}  // namespace

struct ilf_ctx {
  ilf_config cfg;
  Geom g;
  bool is_band = false;
  ilf_band band;
  cudaStream_t stream = nullptr;   // compute stream (kernels)
  cudaStream_t s_up = nullptr;     // host -> device copies
  cudaStream_t s_down = nullptr;   // device -> host copies
  cudaStream_t s_rec = nullptr;    // deblocking record passes (ilf_set_deblock_info): off the upload stream, so copies queued behind one do not wait for it
  // Lanes: a chain over a large batch is dealt to `num_lanes` extra compute streams (ilf_run), so that the drain of one lane's
  // kernel overlaps another lane's kernels; the compute stream joins them (waits for their run events) without holding them up.
  static constexpr int MAX_LANES = 4;
  cudaStream_t lane[MAX_LANES] = {};
  int num_lanes = 1;
  int lane_min_slots = 8;          // batches smaller than this run on the compute stream alone
  std::vector<Slot> slots;
  SlotDev* slots_dev = nullptr;
  size_t plane_y = 0, plane_c = 0, buf_elems = 0;  // elements per plane / per 3-plane buffer
  std::string err;
  long long launches = 0;
  bool timing = false;
  // per-kernel timing (bench.py): event pairs recorded around every launch while timing is on
  struct TimedLaunch { int kernel; cudaEvent_t a, b; };
  std::vector<TimedLaunch> timed;
  std::vector<cudaEvent_t> free_events;
  // run events (fence()): a ring per stream, 0: the compute stream, 1 + i: lane i
  static constexpr int RUN_RING = 64;
  cudaEvent_t run_ring[1 + MAX_LANES][RUN_RING] = {};
  unsigned run_pos[1 + MAX_LANES] = {};
  cudaEvent_t next_run_event(int ring) { return run_ring[ring][run_pos[ring]++ % RUN_RING]; }
  double kernel_ms[ILF_NUM_KERNELS] = {};
  double kernel_bytes[ILF_NUM_KERNELS] = {};
  long long kernel_launches[ILF_NUM_KERNELS] = {};
  int num_ctus = 0;
  CopyPool copy_pool;
  uint32_t* hash_scratch = nullptr;   // ilf_picture_hash
  int* db_work = nullptr;             // tile queues of the deblocking kernel: two ints per stream (the compute stream, then the lanes)
  unsigned long long* search_out = nullptr;   // ilf_deblock_search: [num_slots][ILF_DEBLOCK_SEARCH_MAX][3], allocated by the first search
  cudaEvent_t chunk_ev[COPY_CHUNKS_MAX] = {};   // download: chunk i has reached the staging buffer
  cudaEvent_t ev_caller = nullptr;   // device transfers: the caller's stream up to the call (recorded, then waited for at once)
};

namespace {

int fail(ilf_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

#define CU(ctx, call)                                                                                     \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) return fail(ctx, ILF_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

int check_slot(ilf_ctx* ctx, int slot) {
  if (!ctx) return ILF_ERR_ARG;
  if (slot < 0 || slot >= (int)ctx->slots.size()) return fail(ctx, ILF_ERR_ARG, "slot %d out of range [0,%d)", slot, (int)ctx->slots.size());
  return ILF_OK;
}

int check_range(ilf_ctx* ctx, int first, int n) {
  if (!ctx) return ILF_ERR_ARG;
  if (first < 0 || n < 1 || first + n > (int)ctx->slots.size()) return fail(ctx, ILF_ERR_ARG, "slot range [%d,+%d) out of range", first, n);
  return ILF_OK;
}

// Per-slot ordering.  H2D copies run on the upload stream, kernels on the compute stream or one of its lanes, D2H copies on the
// download stream, so the upload of picture n+1, the filtering of picture n and the download of picture n-1 overlap when the caller
// cycles through several slots.  These events of the slot order the three:
//   ev_up        every H2D copy issued so far for the slot (planes, side information, original, descriptor, halo rows) is done;
//                h2d_pending: such a copy was issued since a compute stream last waited for ev_up.
//   ev_side[k]   the pinned staging region of side-information stage k is free again (the host waits for it before refilling).
//   ev_run       every kernel issued so far on the slot is done: an event of the context's run ring, shared by the slots of one
//                run, recorded on run_stream (the compute stream or a lane; nullptr: no kernel yet).  Copies that overwrite what a
//                kernel reads (uploads, side information, originals, halo rows) and downloads wait for it.
//   ev_down      the last D2H copy of the slot is done (uploads wait for it); d2h_pending: a download was issued since ilf_run last
//                waited for ev_down.
//   ev_rec       the slot's last deblocking record pass (ilf_set_deblock_info, on s_rec after the side-information copies it reads) is
//                done; kernels and the next setter call wait for it while rec_pending.
// A batched entry point validates every slot before it issues anything, then joins each slot to the stream it launches on,
// launches, and fences.

// Orders `st` after the slot's pending upload and, when its last kernels ran on another stream, after them.  Clearing h2d_pending
// is safe because every later kernel of the slot is then ordered after the upload: on `st` by stream order, on another stream
// through the run event that fence() records on `st` after the launches.  The hash and the ALF classification record no run event;
// they synchronise `st` before they return, so the upload is complete.  overwrites_buffers (ilf_run only): the launches write work
// buffers that a download may still read.
int join(ilf_ctx* ctx, Slot& s, cudaStream_t st, bool overwrites_buffers) {
  if (s.h2d_pending) { CU(ctx, cudaStreamWaitEvent(st, s.ev_up, 0)); s.h2d_pending = false; }
  if (s.rec_pending) { CU(ctx, cudaStreamWaitEvent(st, s.ev_rec, 0)); s.rec_pending = false; }
  if (overwrites_buffers && s.d2h_pending) { CU(ctx, cudaStreamWaitEvent(st, s.ev_down, 0)); s.d2h_pending = false; }
  if (s.run_stream && s.run_stream != st) CU(ctx, cudaStreamWaitEvent(st, s.ev_run, 0));
  return ILF_OK;
}

// One event of ring `ring` recorded on `st` becomes ev_run of the slots [first, first + n) (of those with lane_of[i - first] == lane,
// when lane_of is given).  A ring per stream is enough: waiting on an event that was re-recorded on the same stream only waits longer.
int fence(ilf_ctx* ctx, int first, int n, cudaStream_t st, int ring, const uint8_t* lane_of = nullptr, int lane = 0) {
  cudaEvent_t done = ctx->next_run_event(ring);
  CU(ctx, cudaEventRecord(done, st));
  for (int i = 0; i < n; i++)
    if (!lane_of || lane_of[i] == lane) { ctx->slots[first + i].ev_run = done; ctx->slots[first + i].run_stream = st; }
  return ILF_OK;
}

// Control word of a slot's current picture: plane p from buffer result_buf[p] (BatchCtl).
unsigned buf_word(const Slot& s) { return s.result_buf[0] | s.result_buf[1] << 2 | s.result_buf[2] << 4; }

// Compact launch list of the chunk of slots [c0, c0 + cn): grid layer m works on slot c0 + ctl.slot[m] under control word ctl.v[m].
// word(i) gives the control word of slot c0 + i, or < 0 to leave it out; mv_mode >= 0 keeps the slots of that motion-vector
// representation only (none / int16 / int32 are different deblocking search kernels).
template <typename Word>
int compact(const ilf_ctx* ctx, int c0, int cn, int mv_mode, BatchCtl& ctl, Word word) {
  int m = 0;
  for (int i = 0; i < cn; i++) {
    const int v = word(i);
    if (v < 0 || (mv_mode >= 0 && ctx->slots[c0 + i].mv_mode != mv_mode)) continue;
    ctl.v[m] = (uint16_t)v;
    ctl.slot[m++] = (uint8_t)i;
  }
  return m;
}

int timed_collect(ilf_ctx* ctx) {
  if (ctx->timed.empty()) return ILF_OK;
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& t : ctx->timed) {
    float ms = 0;
    CU(ctx, cudaEventElapsedTime(&ms, t.a, t.b));
    ctx->kernel_ms[t.kernel] += ms;
    ctx->kernel_launches[t.kernel]++;
    ctx->free_events.push_back(t.a);
    ctx->free_events.push_back(t.b);
  }
  ctx->timed.clear();
  return ILF_OK;
}

// Opens the event pair around a launch while timing is on (ilf_set_timing / ilf_kernel_times); at most 4096 pairs stay pending.
int timed_begin(ilf_ctx* ctx, int kernel, double algo_bytes) {
  if (ctx->timed.size() >= 4096) if (int rc = timed_collect(ctx)) return rc;
  ctx->kernel_bytes[kernel] += algo_bytes;
  cudaEvent_t ev[2];
  for (int i = 0; i < 2; i++) {
    if (!ctx->free_events.empty()) { ev[i] = ctx->free_events.back(); ctx->free_events.pop_back(); }
    else CU(ctx, cudaEventCreate(&ev[i]));
  }
  ctx->timed.push_back({kernel, ev[0], ev[1]});
  CU(ctx, cudaEventRecord(ev[0], ctx->stream));
  return ILF_OK;
}

// Issues `count` kernels through enqueue() and counts them.  kernel >= 0: while timing is on, an event pair on the compute stream
// brackets them and `bytes` are accounted to that kernel.
template <typename Enqueue>
int launch(ilf_ctx* ctx, int kernel, double bytes, int count, Enqueue enqueue) {
  const bool timed = ctx->timing && kernel >= 0;
  if (timed) if (int rc = timed_begin(ctx, kernel, bytes)) return rc;
  enqueue();
  if (timed) CU(ctx, cudaEventRecord(ctx->timed.back().b, ctx->stream));
  ctx->launches += count;
  CU(ctx, cudaGetLastError());
  return ILF_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup: the library does not link libcuda, so it still
// loads (and exports its symbols) on a machine without a driver.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    cudaDriverEntryPointQueryResult q;
    void* p = nullptr;
    if (cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &p, 12000, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

// Tensor (x, y, z) over `base`: w x h elements of `elem_bytes`, rows `pitch_bytes` apart, `nz` layers `layer_bytes` apart; box bw x bh x 1.
int make_map3(ilf_ctx* ctx, CUtensorMap* out, CUtensorMapDataType dt, void* base, int w, int h, int nz, size_t pitch_bytes, size_t layer_bytes, int bw, int bh);

int16_t* plane_ptr(const ilf_ctx* ctx, const Slot& s, int buf, int plane) {
  int16_t* p = s.planes + (size_t)buf * ctx->buf_elems;
  if (plane >= 1) p += ctx->plane_y;
  if (plane == 2) p += ctx->plane_c;
  return p;
}

// Plane p's part of LOCAL luma rows [first, first + n): width, rows and first row in the plane's samples (chroma halved), pitch.
struct PlaneRows { int w, h, r0, pitch; };
PlaneRows plane_rows(const Geom& g, int p, int first, int n) {
  const int sh = p ? 1 : 0;
  return {g.width >> sh, n >> sh, first >> sh, p ? g.pitch_c : g.pitch_y};
}

int make_map3(ilf_ctx* ctx, CUtensorMap* out, CUtensorMapDataType dt, void* base, int w, int h, int nz, size_t pitch_bytes, size_t layer_bytes, int bw, int bh) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return fail(ctx, ILF_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)nz};
  const cuuint64_t strides[2] = {(cuuint64_t)pitch_bytes, (cuuint64_t)layer_bytes};
  const cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1}, estr[3] = {1, 1, 1};
  const CUresult r = enc(out, dt, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ctx, ILF_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %dx%dx%d tensor, box %dx%d", (int)r, w, h, nz, bw, bh);
  return ILF_OK;
}

// The slot descriptor travels on the upload stream like the side information it points to.
int push_desc(ilf_ctx* ctx, int slot) {
  Slot& s = ctx->slots[slot];
  // the pointers of a slot settle after its first picture: most calls find the device copy up to date
  if (!(s.pushed_valid && memcmp(&s.dev, &s.pushed, sizeof(SlotDev)) == 0)) {
    memcpy(&s.pushed, &s.dev, sizeof(SlotDev));  // padding included, so that the comparison above is exact
    CU(ctx, cudaMemcpyAsync(ctx->slots_dev + slot, &s.pushed, sizeof(SlotDev), cudaMemcpyHostToDevice, ctx->s_up));
    s.pushed_valid = true;
  }
  CU(ctx, cudaEventRecord(s.ev_up, ctx->s_up));
  s.h2d_pending = true;
  return ILF_OK;
}

// What a pointer addresses: cudaMemoryTypeUnregistered (pageable host memory), cudaMemoryTypeHost (page-locked), cudaMemoryTypeDevice
// or cudaMemoryTypeManaged.  `device` (when given) receives the device of device memory.
cudaMemoryType mem_type(const void* p, int* device = nullptr) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return cudaMemoryTypeUnregistered; }
  if (device) *device = at.device;
  return at.type;
}

// Page-locked (cudaHostAlloc / cudaHostRegister / ilf_host_alloc) host memory can be the source or target of an
// asynchronous copy directly; pageable memory goes through the slot's pinned staging buffer.
bool is_pinned(const void* p) { return mem_type(p) == cudaMemoryTypeHost; }

// The host transfers copy with host memcpy or as host <-> device copies: a plane in device memory is refused (its twin is `device_call`).
int refuse_device_planes(ilf_ctx* ctx, const void* y, const void* cb, const void* cr, cudaMemoryType types[3], const char* device_call) {
  const void* planes[3] = {y, cb, cr};
  for (int p = 0; p < 3; p++) {
    types[p] = mem_type(planes[p]);
    if (types[p] == cudaMemoryTypeDevice) return fail(ctx, ILF_ERR_ARG, "plane %d is device memory: use %s", p, device_call);
  }
  return ILF_OK;
}

// A side-information setter stages its arrays between side_begin and side_end: host -> pinned staging region k of the slot ->
// device, asynchronously on the upload stream.
int side_begin(ilf_ctx* ctx, Slot& s, int k, size_t& cursor) {
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  CU(ctx, cudaEventSynchronize(s.ev_side[k]));  // the previous copy out of this staging region is done
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_run, 0));  // kernels of the slot's previous picture may still read the device arrays
  if (s.rec_pending) CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_rec, 0));  // ... and so may its record pass (the grids, motion, slice map)
  cursor = s.side_off[k];
  return ILF_OK;
}

int side_end(ilf_ctx* ctx, int slot, int k) {
  CU(ctx, cudaEventRecord(ctx->slots[slot].ev_side[k], ctx->s_up));
  return push_desc(ctx, slot);
}

// `rows` rows of `row` bytes, dense in the caller's array, `dpitch` bytes apart on the device (0: dense there too).
int stage_side(ilf_ctx* ctx, Slot& s, int k, void* dst, const void* src, size_t row, size_t& cursor, size_t rows = 1, size_t dpitch = 0) {
  const size_t bytes = row * rows;
  const void* from = src;
  if (!(bytes >= 4096 && is_pinned(src))) {  // a page-locked source is copied straight from the caller's array
    if (cursor + bytes > s.side_off[k + 1]) return fail(ctx, ILF_ERR_STATE, "side-information staging overflow");
    memcpy(s.pinned_side + cursor, src, bytes);
    from = s.pinned_side + cursor;
    cursor += (bytes + 255) & ~size_t(255);
  }
  if (!dpitch || dpitch == row) CU(ctx, cudaMemcpyAsync(dst, from, bytes, cudaMemcpyHostToDevice, ctx->s_up));
  else CU(ctx, cudaMemcpy2DAsync(dst, dpitch, from, row, row, rows, cudaMemcpyHostToDevice, ctx->s_up));
  return ILF_OK;
}

struct BandHandle {  // what ilf_band_export writes into ilf_band_handle::opaque
  uint32_t magic;
  int32_t pid, device, width, row0, rows, pitch_y, pitch_c;
  uint64_t plane_y, plane_c, ptr;
  cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(BandHandle) <= sizeof(ilf_band_handle), "ilf_band_handle too small");
constexpr uint32_t BAND_MAGIC = 0x424C4649u;

// Unit grids (deblocking side information, region 0) live on the device with a row pitch of units_pitch elements (multiple of 4);
// the caller's arrays are dense.
int stage_grid(ilf_ctx* ctx, Slot& s, void* dst, const void* src, size_t elem_bytes, size_t& cursor) {
  const Geom& g = ctx->g;
  return stage_side(ctx, s, 0, dst, src, g.units_w * elem_bytes, cursor, g.units_h, g.units_pitch * elem_bytes);
}

int create_impl(ilf_ctx** out, const ilf_config* cfg, const ilf_band* band) {
  if (!out || !cfg) return fail(nullptr, ILF_ERR_ARG, "null argument");
  *out = nullptr;
  if (cfg->width <= 0 || cfg->height <= 0 || (cfg->width & 7) || (cfg->height & 7))
    return fail(nullptr, ILF_ERR_ARG, "picture size %dx%d must be positive multiples of 8", cfg->width, cfg->height);
  if (cfg->width > 16384 || cfg->height > 16384) return fail(nullptr, ILF_ERR_UNSUPPORTED, "picture size %dx%d above 16384", cfg->width, cfg->height);
  if (cfg->bit_depth_luma < 8 || cfg->bit_depth_luma > 12 || cfg->bit_depth_chroma < 8 || cfg->bit_depth_chroma > 12)
    return fail(nullptr, ILF_ERR_ARG, "bit depth must be in 8..12");
  if (cfg->ctu_log2 < 5 || cfg->ctu_log2 > 7) return fail(nullptr, ILF_ERR_ARG, "ctu_log2 must be 5, 6 or 7");
  if (cfg->chroma_format != 1) return fail(nullptr, ILF_ERR_UNSUPPORTED, "only 4:2:0 (chroma_format 1) is supported");
  if (cfg->num_slots < 1) return fail(nullptr, ILF_ERR_ARG, "num_slots must be >= 1");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, ILF_ERR_CUDA, "no CUDA device (%s); libilf_b200 has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, ILF_ERR_ARG, "device %d out of range [0,%d)", cfg->device, ndev);

  ilf_ctx* ctx = new (std::nothrow) ilf_ctx();
  if (!ctx) return fail(nullptr, ILF_ERR_NOMEM, "out of host memory");
  ctx->cfg = *cfg;
  Geom& g = ctx->g;
  g.width = cfg->width; g.height = cfg->height;
  g.ctu_log2 = cfg->ctu_log2;
  const int ctu = 1 << cfg->ctu_log2;
  g.ctus_w = (cfg->width + ctu - 1) >> cfg->ctu_log2;
  g.ctus_h = (cfg->height + ctu - 1) >> cfg->ctu_log2;
  g.bd_luma = cfg->bit_depth_luma; g.bd_chroma = cfg->bit_depth_chroma;
  g.units_w = cfg->width / 4;
  g.row0 = 0; g.rows = cfg->height; g.out_row0 = 0; g.out_rows = cfg->height;
  if (band) {
    if (band->first_ctu_row < 0 || band->num_ctu_rows < 1 || band->first_ctu_row + band->num_ctu_rows > g.ctus_h) {
      delete ctx;
      return fail(nullptr, ILF_ERR_ARG, "band CTU rows [%d,+%d) outside the picture (%d CTU rows)", band->first_ctu_row, band->num_ctu_rows, g.ctus_h);
    }
    ctx->is_band = true;
    ctx->band = *band;
    // luma rows held beyond the band on each side: 4 luma / 3 chroma rows are needed (DESIGN.md); 16 keeps the held region on the
    // 16-luma-row grid of the chroma deblocking edges (8 chroma rows), which the kernels locate by LOCAL row
    const int halo = 16;
    g.out_row0 = band->first_ctu_row << cfg->ctu_log2;
    const int out_end = std::min(cfg->height, (band->first_ctu_row + band->num_ctu_rows) << cfg->ctu_log2);
    g.out_rows = out_end - g.out_row0;
    g.row0 = std::max(0, g.out_row0 - halo);
    g.rows = std::min(cfg->height, out_end + halo) - g.row0;
  }
  g.units_h = g.rows / 4;
  g.units_pitch = (g.units_w + 3) & ~3;
  g.debug = getenv("ILF_DEBUG") ? atoi(getenv("ILF_DEBUG")) : 0;
  g.pitch_y = (cfg->width + 63) & ~63;
  g.pitch_c = (cfg->width / 2 + 63) & ~63;
  ctx->plane_y = (size_t)g.pitch_y * g.rows;
  ctx->plane_c = (size_t)g.pitch_c * (g.rows / 2);
  ctx->buf_elems = ctx->plane_y + 2 * ctx->plane_c;
  ctx->num_ctus = g.ctus_w * g.ctus_h;
  *out = ctx;  // from here on errors are reported through ctx->err and the caller destroys

  CU(ctx, cudaSetDevice(cfg->device));
  CU(ctx, cudaEventCreateWithFlags(&ctx->ev_caller, cudaEventDisableTiming));
  CU(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CU(ctx, cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking));
  CU(ctx, cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking));
  CU(ctx, cudaStreamCreateWithFlags(&ctx->s_rec, cudaStreamNonBlocking));
  ctx->num_lanes = std::max(1, std::min((int)ilf_ctx::MAX_LANES, env_int("ILF_RUN_LANES", 2)));
  ctx->lane_min_slots = std::max(2, env_int("ILF_RUN_LANE_MIN", 8));
  if (ctx->num_lanes > 1)
    for (int i = 0; i < ctx->num_lanes; i++) CU(ctx, cudaStreamCreateWithFlags(&ctx->lane[i], cudaStreamNonBlocking));
  for (auto& ring : ctx->run_ring)
    for (cudaEvent_t& e : ring) CU(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CU(ctx, cudaMalloc(&ctx->db_work, sizeof(int) * 2 * (1 + ilf_ctx::MAX_LANES)));
  CU(ctx, cudaMemset(ctx->db_work, 0, sizeof(int) * 2 * (1 + ilf_ctx::MAX_LANES)));
  ctx->slots.resize(cfg->num_slots);
  CU(ctx, cudaMalloc(&ctx->slots_dev, sizeof(SlotDev) * cfg->num_slots));
  const size_t units = (size_t)g.units_pitch * g.units_h;  // device grids are pitched
  const DbRecLayout rec = db_rec_layout(g);
  for (int i = 0; i < cfg->num_slots; i++) {
    Slot& s = ctx->slots[i];
    CU(ctx, cudaMalloc(&s.planes, 3 * ctx->buf_elems * sizeof(int16_t)));
    CU(ctx, cudaMemsetAsync(s.planes, 0, 3 * ctx->buf_elems * sizeof(int16_t), ctx->s_up));
    CU(ctx, cudaMalloc(&s.info, units * 4));
    CU(ctx, cudaMalloc(&s.info_c, units * 4));
    CU(ctx, cudaMalloc(&s.mv, units * 16));
    CU(ctx, cudaMemsetAsync(s.info, 0, units * 4, ctx->s_up));
    CU(ctx, cudaMemsetAsync(s.info_c, 0, units * 4, ctx->s_up));
    CU(ctx, cudaMemsetAsync(s.mv, 0, units * 16, ctx->s_up));
    CU(ctx, cudaMalloc(&s.db_rec, rec.bytes));
    CU(ctx, cudaMemsetAsync(s.db_rec, 0, rec.bytes, ctx->s_up));
    CU(ctx, cudaMalloc(&s.ctu_slice, ctx->num_ctus));
    CU(ctx, cudaMalloc(&s.db_params, sizeof(ilf_deblock_params)));
    CU(ctx, cudaMalloc(&s.sao, sizeof(ilf_sao_ctu) * ctx->num_ctus));
    CU(ctx, cudaMalloc(&s.alf, sizeof(ilf_alf_params)));
    CU(ctx, cudaMalloc(&s.alf_coef, 25 * 4 * 16 * sizeof(int)));
    CU(ctx, cudaMalloc(&s.alf_coef_dp, ALF_DP_WORDS * sizeof(uint32_t)));
    CU(ctx, cudaMalloc(&s.alf_ctu_enable, 3 * (size_t)ctx->num_ctus));
    CU(ctx, cudaMalloc(&s.alf_class, units));
    auto up256 = [](size_t v) { return (v + 255) & ~size_t(255); };
    s.side_off[0] = 0;
    s.side_off[1] = up256(sizeof(ilf_deblock_params)) + 2 * up256(units * 4) + up256(units * 16) + up256(ctx->num_ctus);
    s.side_off[2] = s.side_off[1] + up256(sizeof(ilf_sao_ctu) * ctx->num_ctus);
    s.side_off[3] = s.side_off[2] + up256(sizeof(ilf_alf_params)) + up256(3 * (size_t)ctx->num_ctus) + up256(25 * 4 * 16 * sizeof(int)) + up256(ALF_DP_WORDS * sizeof(uint32_t));
    s.pinned_side_bytes = s.side_off[3];
    CU(ctx, cudaMallocHost(&s.pinned_side, s.pinned_side_bytes));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_up, cudaEventDisableTiming));
    s.ev_run = ctx->run_ring[0][0];  // never recorded yet: waiting on it is a no-op
    CU(ctx, cudaEventCreateWithFlags(&s.ev_down, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&s.ev_rec, cudaEventDisableTiming));
    for (int k = 0; k < 3; k++) CU(ctx, cudaEventCreateWithFlags(&s.ev_side[k], cudaEventDisableTiming));
    memset(&s.dev, 0, sizeof(s.dev));
    for (int b = 0; b < 3; b++)
      for (int p = 0; p < 3; p++) s.dev.buf[b][p] = plane_ptr(ctx, s, b, p);
    s.dev.alf_class = s.alf_class;
    {
      const size_t grid_bytes = units * 4;
      if (int rc = make_map3(ctx, &s.dev.tm_info, CU_TENSOR_MAP_DATA_TYPE_UINT32, s.info, g.units_w, g.units_h, 1, (size_t)g.units_pitch * 4, grid_bytes, DB_BOX_UNITS, 8)) return rc;
      if (int rc = make_map3(ctx, &s.dev.tm_info_c, CU_TENSOR_MAP_DATA_TYPE_UINT32, s.info_c, g.units_w, g.units_h, 1, (size_t)g.units_pitch * 4, grid_bytes, DB_BOX_UNITS, 8)) return rc;
      if (int rc = make_map3(ctx, &s.dev.tm_mv16, CU_TENSOR_MAP_DATA_TYPE_UINT32, s.mv, g.units_w * 2, g.units_h, 1, (size_t)g.units_pitch * 8, units * 8, DB_BOX_MV16_WORDS, 8)) return rc;
      if (int rc = make_map3(ctx, &s.dev.tm_mv32, CU_TENSOR_MAP_DATA_TYPE_UINT32, s.mv, g.units_w * 4, g.units_h, 1, (size_t)g.units_pitch * 16, units * 16, DB_BOX_MV32_WORDS, 8)) return rc;
      const int box_w[DB_REC_KINDS] = {DB_REC_LV_W, DB_REC_LH_W, DB_REC_CV_W, DB_REC_CH_W}, box_h[DB_REC_KINDS] = {DB_REC_LV_H, DB_REC_LH_H, DB_REC_CV_H, DB_REC_CH_H};
      for (int k = 0; k < DB_REC_KINDS; k++)
        if (int rc = make_map3(ctx, &s.dev.tm_rec[k], rec.elem[k] == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT32, static_cast<char*>(s.db_rec) + rec.off[k],
                               rec.cols[k], rec.rows[k], 1, (size_t)rec.pitch[k] * rec.elem[k], (size_t)rec.pitch[k] * rec.elem[k] * rec.rows[k], box_w[k], box_h[k]))
          return rc;
    }
    for (int p = 0; p < 3; p++) {
      const PlaneRows pr = plane_rows(g, p, 0, g.rows);
      if (int rc = make_map3(ctx, &s.dev.tm_db[p], CU_TENSOR_MAP_DATA_TYPE_UINT16, plane_ptr(ctx, s, 0, p), pr.w, pr.h, 3, (size_t)pr.pitch * 2, ctx->buf_elems * 2, p ? DB_BOX_CW : DB_BOX_W,
                             p ? DB_BAND_ROWS / 2 : DB_BAND_ROWS))
        return rc;
      if (int rc = make_map3(ctx, &s.dev.tm_sao[p], CU_TENSOR_MAP_DATA_TYPE_UINT16, plane_ptr(ctx, s, 0, p), pr.w, pr.h, 3, (size_t)pr.pitch * 2, ctx->buf_elems * 2, SAO_TILE,
                             SAO_BAND_ROWS + 2))
        return rc;
      if (int rc = make_map3(ctx, &s.dev.tm_alf[p], CU_TENSOR_MAP_DATA_TYPE_UINT16, plane_ptr(ctx, s, 0, p), pr.w, pr.h, 3, (size_t)pr.pitch * 2, ctx->buf_elems * 2, ALF_TILE + 16,
                             ALF_BAND_ROWS + 2 * (p ? ALF_HALO_C : ALF_HALO_Y)))
        return rc;
    }
    if (int rc = push_desc(ctx, i)) return rc;
  }
  CU(ctx, cudaStreamSynchronize(ctx->s_up));
  for (Slot& s : ctx->slots) s.h2d_pending = false;
  return ILF_OK;
}

int sync_all(ilf_ctx* ctx) {
  CU(ctx, cudaStreamSynchronize(ctx->s_up));
  CU(ctx, cudaStreamSynchronize(ctx->s_rec));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->s_down));
  return ILF_OK;
}

}  // namespace

extern "C" {

int ilf_abi_version(void) { return ILF_ABI_VERSION; }

int ilf_create(ilf_ctx** out, const ilf_config* cfg) {
  int rc = create_impl(out, cfg, nullptr);
  if (rc != ILF_OK && out && *out) { g_create_error = (*out)->err; ilf_destroy(*out); *out = nullptr; }
  return rc;
}

int ilf_create_band(ilf_ctx** out, const ilf_config* cfg, const ilf_band* band) {
  if (!band) return fail(nullptr, ILF_ERR_ARG, "null band");
  int rc = create_impl(out, cfg, band);
  if (rc != ILF_OK && out && *out) { g_create_error = (*out)->err; ilf_destroy(*out); *out = nullptr; }
  return rc;
}

int ilf_destroy(ilf_ctx* ctx) {
  if (!ctx) return ILF_OK;
  cudaSetDevice(ctx->cfg.device);
  const auto streams = {ctx->s_up, ctx->s_rec, ctx->stream, ctx->s_down, ctx->lane[0], ctx->lane[1], ctx->lane[2], ctx->lane[3]};
  for (cudaStream_t st : streams) if (st) cudaStreamSynchronize(st);
  for (Slot& s : ctx->slots) {
    for (auto& nb : s.nb) if (nb.ipc_base) cudaIpcCloseMemHandle(nb.ipc_base);
    cudaFree(s.planes); cudaFree(s.info); cudaFree(s.info_c); cudaFree(s.mv); cudaFree(s.db_rec); cudaFree(s.ctu_slice); cudaFree(s.db_params);
    cudaFree(s.sao); cudaFree(s.alf); cudaFree(s.alf_coef); cudaFree(s.alf_coef_dp); cudaFree(s.alf_ctu_enable); cudaFree(s.alf_class);
    cudaFree(s.org); cudaFree(s.stats_avail); cudaFree(s.stats); cudaFree(s.alf_stats);
    if (s.pinned) cudaFreeHost(s.pinned);
    if (s.pinned_down) cudaFreeHost(s.pinned_down);
    if (s.pinned_side) cudaFreeHost(s.pinned_side);
    for (cudaEvent_t e : {s.ev_up, s.ev_down, s.ev_rec, s.ev_side[0], s.ev_side[1], s.ev_side[2]}) if (e) cudaEventDestroy(e);
  }
  for (auto& ring : ctx->run_ring)
    for (cudaEvent_t e : ring) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->chunk_ev) if (e) cudaEventDestroy(e);
  if (ctx->ev_caller) cudaEventDestroy(ctx->ev_caller);
  cudaFree(ctx->slots_dev);
  cudaFree(ctx->hash_scratch);
  cudaFree(ctx->db_work);
  cudaFree(ctx->search_out);
  for (auto& t : ctx->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
  for (cudaEvent_t e : ctx->free_events) cudaEventDestroy(e);
  for (cudaStream_t st : streams) if (st) cudaStreamDestroy(st);
  delete ctx;
  return ILF_OK;
}

const char* ilf_last_error(const ilf_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int ilf_get_config(const ilf_ctx* ctx, ilf_config* out) {
  if (!ctx || !out) return ILF_ERR_ARG;
  *out = ctx->cfg;
  return ILF_OK;
}

int ilf_get_band(const ilf_ctx* ctx, ilf_band* out, int32_t* first_row, int32_t* num_rows) {
  if (!ctx) return ILF_ERR_ARG;
  if (out) { if (ctx->is_band) *out = ctx->band; else { out->first_ctu_row = 0; out->num_ctu_rows = ctx->g.ctus_h; } }
  if (first_row) *first_row = ctx->g.row0;
  if (num_rows) *num_rows = ctx->g.rows;
  return ILF_OK;
}

// Row chunks of a staged transfer of LOCAL luma rows [first, first + n): luma in up to 8 pieces, each chroma plane in up to 2
// (about 2 MB each for a 4K picture).
static int make_chunks(const Geom& g, int first, int n, CopyChunk* out) {
  int k = 0;
  size_t off = 0;
  for (int p = 0; p < 3; p++) {
    const PlaneRows pr = plane_rows(g, p, first, n);
    const int pieces = std::max(1, std::min(p ? 2 : 8, pr.h / 64));
    for (int i = 0; i < pieces; i++) {
      const int a = (int)((long long)pr.h * i / pieces), b = (int)((long long)pr.h * (i + 1) / pieces);
      out[k++] = {p, pr.r0 + a, b - a, off + (size_t)a * pr.w};
    }
    off += (size_t)pr.w * pr.h;
  }
  return k;
}

// The state changes of a transfer, shared by the host calls and the device calls (ilf_*_device).
// Before a new picture is written into buffer 0: that buffer may still be read by kernels of the slot's previous picture, or by its
// download when no stage ran on a plane.
static int upload_begin(ilf_ctx* ctx, Slot& s) {
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_run, 0));
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_down, 0));
  return ILF_OK;
}

// After the copies of a new picture are issued on the upload stream: the side information must be set again, the original is
// stale for the deblocking search, and every plane's current picture is the upload.
static int upload_end(ilf_ctx* ctx, Slot& s) {
  CU(ctx, cudaEventRecord(s.ev_up, ctx->s_up));
  s.h2d_pending = true;
  s.uploaded = true;
  s.has_db = s.has_sao = s.has_alf = false;
  s.org_since_upload = false;
  s.result_buf[0] = s.result_buf[1] = s.result_buf[2] = 0;
  return ILF_OK;
}

// A download reads each plane's current buffer: after the slot's last kernels, and after its upload when no stage ran on a plane.
static int download_begin(ilf_ctx* ctx, Slot& s) {
  CU(ctx, cudaStreamWaitEvent(ctx->s_down, s.ev_run, 0));
  CU(ctx, cudaStreamWaitEvent(ctx->s_down, s.ev_up, 0));
  return ILF_OK;
}

// An asynchronous download is pending: ilf_wait waits for it, the slot's next run and upload are ordered after it.
static int download_end(ilf_ctx* ctx, Slot& s) {
  CU(ctx, cudaEventRecord(s.ev_down, ctx->s_down));
  s.d2h_pending = true;
  return ILF_OK;
}

// Copies host rows [first, first + n) (LOCAL luma rows of the held region; chroma rows first/2 ..) into the slot's input buffer.
static int upload_rows(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr, int first, int n) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!y || !cb || !cr) return fail(ctx, ILF_ERR_ARG, "null plane pointer");
  cudaMemoryType types[3];
  if (int rc = refuse_device_planes(ctx, y, cb, cr, types, "ilf_upload_device")) return rc;
  Slot& s = ctx->slots[slot];
  const Geom& g = ctx->g;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = upload_begin(ctx, s)) return rc;
  const int16_t* srcs[3] = {y, cb, cr};
  const ptrdiff_t strides[3] = {sy, scb, scr};
  if (types[0] == cudaMemoryTypeHost && types[1] == cudaMemoryTypeHost && types[2] == cudaMemoryTypeHost) {
    for (int p = 0; p < 3; p++) {
      const PlaneRows pr = plane_rows(g, p, first, n);
      CU(ctx, cudaMemcpy2DAsync(plane_ptr(ctx, s, 0, p) + (size_t)pr.r0 * pr.pitch, (size_t)pr.pitch * 2, srcs[p], (size_t)strides[p] * 2, (size_t)pr.w * 2, pr.h, cudaMemcpyHostToDevice, ctx->s_up));
    }
  } else {
    if (!s.pinned) CU(ctx, cudaMallocHost(&s.pinned, ctx->buf_elems * sizeof(int16_t)));
    CU(ctx, cudaEventSynchronize(s.ev_up));    // staging buffer: the previous staged upload has been consumed
    // helper threads fill the staging buffer chunk by chunk; this thread hands every finished chunk to the DMA engine, in order
    CopyChunk ch[COPY_CHUNKS_MAX];
    const int nch = make_chunks(g, first, n, ch);
    std::atomic<int> ready[COPY_CHUNKS_MAX];
    for (int i = 0; i < nch; i++) ready[i].store(0, std::memory_order_relaxed);
    int16_t* stage = s.pinned;
    auto copy = [&, stage](int i) {
      const CopyChunk& c = ch[i];
      const PlaneRows pr = plane_rows(g, c.plane, first, n);
      const int16_t* src = srcs[c.plane] + (ptrdiff_t)(c.row0 - pr.r0) * strides[c.plane];
      int16_t* d = stage + c.stage_off;
      for (int r = 0; r < c.rows; r++) memcpy(d + (size_t)r * pr.w, src + (ptrdiff_t)r * strides[c.plane], (size_t)pr.w * 2);
      ready[i].store(1, std::memory_order_release);
    };
    const bool par = ctx->copy_pool.threads() > 1 && nch > 1;
    if (par) ctx->copy_pool.start(nch, copy);
    cudaError_t err = cudaSuccess;
    for (int i = 0; i < nch; i++) {
      if (par) while (!ready[i].load(std::memory_order_acquire)) std::this_thread::yield();
      else copy(i);
      const CopyChunk& c = ch[i];
      const PlaneRows pr = plane_rows(g, c.plane, first, n);
      const cudaError_t e = cudaMemcpy2DAsync(plane_ptr(ctx, s, 0, c.plane) + (size_t)c.row0 * pr.pitch, (size_t)pr.pitch * 2, stage + c.stage_off, (size_t)pr.w * 2, (size_t)pr.w * 2,
                                              c.rows, cudaMemcpyHostToDevice, ctx->s_up);
      if (e != cudaSuccess && err == cudaSuccess) err = e;
    }
    if (par) ctx->copy_pool.wait();
    CU(ctx, err);
  }
  return upload_end(ctx, s);
}

// Host planes cover the rows the context HOLDS: the whole picture, or for a band context picture rows
// [row0, row0 + rows) as reported by ilf_get_band (pointer = first held row).
int ilf_upload(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr) {
  if (!ctx) return ILF_ERR_ARG;
  return upload_rows(ctx, slot, y, sy, cb, scb, cr, scr, 0, ctx->g.rows);
}

// Host planes cover the band's OWN rows (ilf_get_band_rows); the halo rows come from the neighbours (ilf_band_exchange).
int ilf_upload_band(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr) {
  if (!ctx) return ILF_ERR_ARG;
  return upload_rows(ctx, slot, y, sy, cb, scb, cr, scr, ctx->g.out_row0 - ctx->g.row0, ctx->g.out_rows);
}

// Issues the device -> host copy of LOCAL rows [first, first + n) of the slot's current picture.  Into page-locked memory
// the copy is asynchronous (ilf_wait / ilf_sync complete it); into pageable memory the call stages and blocks.
static int download_rows(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr, int first, int n) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!y || !cb || !cr) return fail(ctx, ILF_ERR_ARG, "null plane pointer");
  cudaMemoryType types[3];
  if (int rc = refuse_device_planes(ctx, y, cb, cr, types, "ilf_download_device")) return rc;
  Slot& s = ctx->slots[slot];
  if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: download before upload", slot);
  const Geom& g = ctx->g;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = download_begin(ctx, s)) return rc;
  int16_t* dsts[3] = {y, cb, cr};
  const ptrdiff_t strides[3] = {sy, scb, scr};
  if (types[0] == cudaMemoryTypeHost && types[1] == cudaMemoryTypeHost && types[2] == cudaMemoryTypeHost) {
    for (int p = 0; p < 3; p++) {
      const PlaneRows pr = plane_rows(g, p, first, n);
      CU(ctx, cudaMemcpy2DAsync(dsts[p], (size_t)strides[p] * 2, plane_ptr(ctx, s, s.result_buf[p], p) + (size_t)pr.r0 * pr.pitch, (size_t)pr.pitch * 2, (size_t)pr.w * 2, pr.h, cudaMemcpyDeviceToHost, ctx->s_down));
    }
    return download_end(ctx, s);
  }
  // staged: the DMA engine delivers row chunks into the page-locked buffer, helper threads (and this one) copy every chunk on to
  // the caller's planes as soon as its event has fired
  if (!s.pinned_down) CU(ctx, cudaMallocHost(&s.pinned_down, ctx->buf_elems * sizeof(int16_t)));
  CopyChunk ch[COPY_CHUNKS_MAX];
  const int nch = make_chunks(g, first, n, ch);
  int16_t* stage = s.pinned_down;
  for (int i = 0; i < nch; i++) {
    const CopyChunk& c = ch[i];
    const PlaneRows pr = plane_rows(g, c.plane, first, n);
    if (!ctx->chunk_ev[i]) CU(ctx, cudaEventCreateWithFlags(&ctx->chunk_ev[i], cudaEventDisableTiming));
    CU(ctx, cudaMemcpy2DAsync(stage + c.stage_off, (size_t)pr.w * 2, plane_ptr(ctx, s, s.result_buf[c.plane], c.plane) + (size_t)c.row0 * pr.pitch, (size_t)pr.pitch * 2,
                              (size_t)pr.w * 2, c.rows, cudaMemcpyDeviceToHost, ctx->s_down));
    CU(ctx, cudaEventRecord(ctx->chunk_ev[i], ctx->s_down));
  }
  CU(ctx, cudaEventRecord(s.ev_down, ctx->s_down));
  std::atomic<int> failed(0);
  const int device = ctx->cfg.device;
  auto copy = [&, stage, device](int i) {
    const CopyChunk& c = ch[i];
    cudaSetDevice(device);
    if (cudaEventSynchronize(ctx->chunk_ev[i]) != cudaSuccess) { failed.store(1); return; }
    const PlaneRows pr = plane_rows(g, c.plane, first, n);
    int16_t* d = dsts[c.plane] + (ptrdiff_t)(c.row0 - pr.r0) * strides[c.plane];
    const int16_t* src = stage + c.stage_off;
    for (int r = 0; r < c.rows; r++) memcpy(d + (ptrdiff_t)r * strides[c.plane], src + (size_t)r * pr.w, (size_t)pr.w * 2);
  };
  if (ctx->copy_pool.threads() > 1 && nch > 1) { ctx->copy_pool.start(nch, copy); ctx->copy_pool.wait(); }
  else for (int i = 0; i < nch; i++) copy(i);
  if (failed.load()) return fail(ctx, ILF_ERR_CUDA, "device -> host copy failed: %s", cudaGetErrorString(cudaGetLastError()));
  return ILF_OK;  // synchronous: nothing left pending
}

int ilf_download_async(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr) {
  if (!ctx) return ILF_ERR_ARG;
  return download_rows(ctx, slot, y, sy, cb, scb, cr, scr, 0, ctx->g.rows);
}

int ilf_download_band(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr) {
  if (!ctx) return ILF_ERR_ARG;
  if (int rc = download_rows(ctx, slot, y, sy, cb, scb, cr, scr, ctx->g.out_row0 - ctx->g.row0, ctx->g.out_rows)) return rc;
  return ilf_wait(ctx, slot);
}

int ilf_get_band_rows(const ilf_ctx* ctx, int32_t* own_first, int32_t* own_rows) {
  if (!ctx) return ILF_ERR_ARG;
  if (own_first) *own_first = ctx->g.out_row0;
  if (own_rows) *own_rows = ctx->g.out_rows;
  return ILF_OK;
}

int ilf_band_export(ilf_ctx* ctx, int slot, ilf_band_handle* out) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null handle");
  Slot& s = ctx->slots[slot];
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  BandHandle h;
  memset(&h, 0, sizeof(h));
  h.magic = BAND_MAGIC; h.pid = (int32_t)getpid(); h.device = ctx->cfg.device; h.width = ctx->g.width;
  h.row0 = ctx->g.row0; h.rows = ctx->g.rows; h.pitch_y = ctx->g.pitch_y; h.pitch_c = ctx->g.pitch_c;
  h.plane_y = ctx->plane_y; h.plane_c = ctx->plane_c; h.ptr = (uint64_t)(uintptr_t)s.planes;
  CU(ctx, cudaIpcGetMemHandle(&h.ipc, s.planes));
  memset(out, 0, sizeof(*out));
  memcpy(out->opaque, &h, sizeof(h));
  return ILF_OK;
}

int ilf_band_connect(ilf_ctx* ctx, int slot, int side, const ilf_band_handle* neighbour) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!neighbour || (side != ILF_BAND_ABOVE && side != ILF_BAND_BELOW)) return fail(ctx, ILF_ERR_ARG, "bad neighbour handle or side");
  BandHandle h;
  memcpy(&h, neighbour->opaque, sizeof(h));
  if (h.magic != BAND_MAGIC || h.width != ctx->g.width) return fail(ctx, ILF_ERR_ARG, "neighbour handle does not describe a band of this picture");
  Slot& s = ctx->slots[slot];
  Slot::Neighbour& nb = s.nb[side];
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (nb.ipc_base) { cudaIpcCloseMemHandle(nb.ipc_base); nb.ipc_base = nullptr; }
  if (h.pid == (int32_t)getpid()) {
    if (h.device != ctx->cfg.device) {
      int can = 0;
      CU(ctx, cudaDeviceCanAccessPeer(&can, ctx->cfg.device, h.device));
      if (can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(h.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctx, ILF_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) failed: %s", h.device, cudaGetErrorString(e));
        cudaGetLastError();
      } else {
        // the halo kernel dereferences the neighbour's pointer: without a peer mapping that is an illegal address, not a slow path
        return fail(ctx, ILF_ERR_UNSUPPORTED, "no peer access from device %d to device %d: band mode needs NVLink / PCIe P2P between neighbouring bands", ctx->cfg.device, h.device);
      }
    }
    nb.planes = (const int16_t*)(uintptr_t)h.ptr;
  } else {
    void* base = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&base, h.ipc, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(ctx, ILF_ERR_CUDA, "cudaIpcOpenMemHandle failed: %s (no P2P path to device %d?)", cudaGetErrorString(e), h.device);
    nb.ipc_base = base;
    nb.planes = (const int16_t*)base;
  }
  nb.device = h.device; nb.row0 = h.row0; nb.rows = h.rows; nb.pitch_y = h.pitch_y; nb.pitch_c = h.pitch_c; nb.plane_y = (size_t)h.plane_y; nb.plane_c = (size_t)h.plane_c;
  return ILF_OK;
}

// Halo rows come over NVLink with ONE kernel per call: every CTA row copies one (slot, side, plane) strip out of the
// neighbour's input buffer (a peer or IPC-mapped pointer) with 8-byte loads and stores.  A strip is a few rows of a plane, so
// a copy-engine transfer per strip (six per slot) costs more in launch latency than in bytes.
namespace {
struct HaloCopy { const int16_t* src; int16_t* dst; int src_pitch, dst_pitch, words, rows; };  // pitches in samples, words of 8 bytes per row
constexpr int HALO_MAX = 96;
struct HaloBatch { HaloCopy c[HALO_MAX]; };
__global__ void __launch_bounds__(256) band_halo_kernel(HaloBatch hb) {
  const HaloCopy& h = hb.c[blockIdx.y];
  const int total = h.words * h.rows;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / h.words, x = i - r * h.words;
    reinterpret_cast<uint2*>(h.dst + (size_t)r * h.dst_pitch)[x] = reinterpret_cast<const uint2*>(h.src + (size_t)r * h.src_pitch)[x];
  }
}
}  // namespace

int ilf_band_exchange_batch(ilf_ctx* ctx, int first_slot, int num_slots) {
  if (int rc = check_range(ctx, first_slot, num_slots)) return rc;
  if (!ctx->is_band) return fail(ctx, ILF_ERR_STATE, "not a band context");
  const Geom& g = ctx->g;
  // picture rows [h0, h1) of the halo above (side 0) and below (side 1); empty at a picture border
  const int h0[2] = {g.row0, g.out_row0 + g.out_rows}, h1[2] = {g.out_row0, g.row0 + g.rows};
  for (int slot = first_slot; slot < first_slot + num_slots; slot++)
    for (int side = 0; side < 2; side++) {
      const Slot::Neighbour& nb = ctx->slots[slot].nb[side];
      if (h1[side] <= h0[side]) continue;
      if (!nb.planes) return fail(ctx, ILF_ERR_STATE, "slot %d: no neighbour connected %s the band", slot, side == ILF_BAND_ABOVE ? "above" : "below");
      if (h0[side] < nb.row0 || h1[side] > nb.row0 + nb.rows) return fail(ctx, ILF_ERR_ARG, "neighbour band does not hold picture rows [%d,%d)", h0[side], h1[side]);
    }
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  HaloBatch hb;
  int n = 0;
  auto flush = [&]() -> int {
    const int rc = n ? launch(ctx, -1, 0, 1, [&] { band_halo_kernel<<<dim3(8, n), 256, 0, ctx->s_up>>>(hb); }) : ILF_OK;
    n = 0;
    return rc;
  };
  for (int slot = first_slot; slot < first_slot + num_slots; slot++) {
    Slot& s = ctx->slots[slot];
    CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_run, 0));  // kernels of the slot's previous run may still read the halo rows
    for (int side = 0; side < 2; side++) {
      if (h1[side] <= h0[side]) continue;
      const Slot::Neighbour& nb = s.nb[side];
      for (int p = 0; p < 3; p++) {
        const PlaneRows pr = plane_rows(g, p, h0[side] - g.row0, h1[side] - h0[side]);
        const int npitch = p ? nb.pitch_c : nb.pitch_y;
        if (n == HALO_MAX) if (int rc = flush()) return rc;
        HaloCopy& c = hb.c[n++];
        c.src = nb.planes + (p >= 1 ? nb.plane_y : 0) + (p == 2 ? nb.plane_c : 0) + (size_t)((h0[side] - nb.row0) >> (p ? 1 : 0)) * npitch;  // neighbour's input buffer (buffer 0)
        c.dst = plane_ptr(ctx, s, 0, p) + (size_t)pr.r0 * pr.pitch;
        c.src_pitch = npitch; c.dst_pitch = pr.pitch;
        c.words = (pr.w * 2) / 8;   // widths are multiples of 8 luma / 4 chroma samples
        c.rows = pr.h;
      }
    }
  }
  if (int rc = flush()) return rc;
  for (int slot = first_slot; slot < first_slot + num_slots; slot++) {
    Slot& s = ctx->slots[slot];
    CU(ctx, cudaEventRecord(s.ev_up, ctx->s_up));
    s.h2d_pending = true;
  }
  return ILF_OK;
}

int ilf_band_exchange(ilf_ctx* ctx, int slot) {
  if (int rc = check_slot(ctx, slot)) return rc;
  return ilf_band_exchange_batch(ctx, slot, 1);
}

// Decoded-picture hash of the slot's current picture, computed where the picture is (ilf_hash.cu).
// The slot's current planes for a hash, with the compute stream joined to the slot.
static int hash_planes(ilf_ctx* ctx, Slot& s, const int16_t* planes[3]) {
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (!ctx->hash_scratch) CU(ctx, cudaMalloc(&ctx->hash_scratch, (6 * 16384 + 8) * sizeof(uint32_t)));
  if (int rc = join(ctx, s, ctx->stream, false)) return rc;
  for (int p = 0; p < 3; p++) planes[p] = plane_ptr(ctx, s, s.result_buf[p], p);
  return ILF_OK;
}

int ilf_picture_hash(ilf_ctx* ctx, int slot, int kind, uint32_t out[3]) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out || (kind != ILF_HASH_CRC && kind != ILF_HASH_CHECKSUM)) return fail(ctx, ILF_ERR_ARG, "bad hash kind or null output");
  if (ctx->is_band) return fail(ctx, ILF_ERR_STATE, "a band context holds a part of the picture only");
  Slot& s = ctx->slots[slot];
  if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: hash before upload", slot);
  const int16_t* planes[3];
  if (int rc = hash_planes(ctx, s, planes)) return rc;
  uint32_t crc[3], sum[3];
  cudaError_t e = cudaSuccess;
  if (int rc = launch(ctx, -1, 0, 2, [&] { e = picture_hash(ctx->g, planes, ctx->hash_scratch, ctx->stream, crc, sum); })) return rc;
  CU(ctx, e);
  for (int p = 0; p < 3; p++) out[p] = kind == ILF_HASH_CRC ? crc[p] : sum[p];
  return ILF_OK;
}

// The band's own rows as a part of the picture's hash (ilf_hash_combine in ilf_hash.cu folds the parts).
int ilf_picture_hash_band(ilf_ctx* ctx, int slot, ilf_hash_part* out) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null output");
  if (!ctx->is_band) return fail(ctx, ILF_ERR_STATE, "not a band context (ilf_picture_hash hashes the whole picture)");
  Slot& s = ctx->slots[slot];
  if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: hash before upload", slot);
  const int16_t* planes[3];
  if (int rc = hash_planes(ctx, s, planes)) return rc;
  const Geom& g = ctx->g;
  ilf_hash_part part;
  memset(&part, 0, sizeof(part));
  part.width = g.width; part.height = g.height; part.bd_luma = g.bd_luma; part.bd_chroma = g.bd_chroma;
  part.first_row = g.out_row0; part.num_rows = g.out_rows;
  cudaError_t e = cudaSuccess;
  if (int rc = launch(ctx, -1, 0, 2, [&] { e = hash_rows(g, planes, ctx->hash_scratch, ctx->stream, g.out_row0 - g.row0, g.out_rows, g.out_row0, part.crc, part.sum); })) return rc;
  CU(ctx, e);
  *out = part;
  return ILF_OK;
}

// Reference border extension on the way down (Picture::extendPicBorder, Picture.cpp:996-1040): the planes are downloaded into buffers
// that have `margin` luma (margin / 2 chroma) samples of room on every side, and the margins are filled by replication -- rows by
// the copy threads, so the decoder's own extendPicBorder pass over the picture is not needed any more.
// Fills the left / right margins of the n luma rows (n / 2 chroma rows) the plane pointers start at, and the margin rows above the
// first row (with the corners) when `top`, those below the last row when `bottom`.
static void extend_margins(ilf_ctx* ctx, int16_t* const planes[3], const ptrdiff_t strides[3], int margin, int n, bool top, bool bottom) {
  const Geom& g = ctx->g;
  // left / right margins of every row, in the row chunks of a staged transfer on the copy threads; then the top / bottom rows
  // (which include the corners)
  CopyChunk ch[COPY_CHUNKS_MAX];
  const int nch = make_chunks(g, 0, n, ch);
  auto sides = [&](int i) {
    const CopyChunk& c = ch[i];
    const int w = plane_rows(g, c.plane, 0, n).w, m = c.plane ? margin / 2 : margin;
    for (int r = c.row0; r < c.row0 + c.rows; r++) {
      int16_t* row = planes[c.plane] + (ptrdiff_t)r * strides[c.plane];
      const int16_t a = row[0], b = row[w - 1];
      for (int x = 0; x < m; x++) { row[-m + x] = a; row[w + x] = b; }
    }
  };
  if (ctx->copy_pool.threads() > 1) { ctx->copy_pool.start(nch, sides); ctx->copy_pool.wait(); }
  else for (int i = 0; i < nch; i++) sides(i);
  for (int p = 0; p < 3; p++) {
    const PlaneRows pr = plane_rows(g, p, 0, n);
    const int w = pr.w, m = p ? margin / 2 : margin;
    int16_t* first = planes[p] - m;
    int16_t* last = planes[p] + (ptrdiff_t)(pr.h - 1) * strides[p] - m;
    for (int r = 1; r <= m; r++) {
      if (top) memcpy(first - (ptrdiff_t)r * strides[p], first, sizeof(int16_t) * (size_t)(w + 2 * m));
      if (bottom) memcpy(last + (ptrdiff_t)r * strides[p], last, sizeof(int16_t) * (size_t)(w + 2 * m));
    }
  }
}

int ilf_download_extended(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr, int margin) {
  if (margin < 0 || (margin & 1)) return fail(ctx, ILF_ERR_ARG, "margin must be even and >= 0");
  if (ctx && ctx->is_band) return fail(ctx, ILF_ERR_STATE, "not available on band contexts");
  if (int rc = ilf_download(ctx, slot, y, sy, cb, scb, cr, scr)) return rc;
  int16_t* const planes[3] = {y, cb, cr};
  const ptrdiff_t strides[3] = {sy, scb, scr};
  extend_margins(ctx, planes, strides, margin, ctx->g.height, true, true);
  return ILF_OK;
}

// The band's own rows and their margins; the rows above / below the picture only from the band that owns its first / last row.
int ilf_download_band_extended(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr, int margin) {
  if (margin < 0 || (margin & 1)) return fail(ctx, ILF_ERR_ARG, "margin must be even and >= 0");
  if (ctx && !ctx->is_band) return fail(ctx, ILF_ERR_STATE, "not a band context (ilf_download_extended downloads the whole picture)");
  if (int rc = ilf_download_band(ctx, slot, y, sy, cb, scb, cr, scr)) return rc;
  const Geom& g = ctx->g;
  int16_t* const planes[3] = {y, cb, cr};
  const ptrdiff_t strides[3] = {sy, scb, scr};
  extend_margins(ctx, planes, strides, margin, g.out_rows, g.out_row0 == 0, g.out_row0 + g.out_rows == g.height);
  return ILF_OK;
}

int ilf_wait(ilf_ctx* ctx, int slot) {
  if (int rc = check_slot(ctx, slot)) return rc;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  CU(ctx, cudaEventSynchronize(ctx->slots[slot].ev_down));
  return ILF_OK;
}

int ilf_download(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t sy, int16_t* cb, ptrdiff_t scb, int16_t* cr, ptrdiff_t scr) {
  if (int rc = ilf_download_async(ctx, slot, y, sy, cb, scb, cr, scr)) return rc;
  return ilf_wait(ctx, slot);
}

int ilf_sync(ilf_ctx* ctx) {
  if (!ctx) return ILF_ERR_ARG;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  return sync_all(ctx);
}

void* ilf_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void ilf_host_free(void* p) { if (p) cudaFreeHost(p); }
int ilf_host_register(void* p, size_t bytes) { if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) != cudaSuccess) { cudaGetLastError(); return ILF_ERR_CUDA; } return ILF_OK; }
int ilf_host_unregister(void* p) { if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return ILF_ERR_CUDA; } return ILF_OK; }

// Whether any of the n units of a dense grid is intra, in 64-bit words, a cache line at a time, stopping at the first hit.
static bool any_intra(const uint32_t* grid, size_t n) {
  constexpr uint64_t mask = ILF_BI_INTRA | (uint64_t)ILF_BI_INTRA << 32;
  size_t i = 0;
  for (; i + 16 <= n; i += 16) {
    uint64_t w[8];
    memcpy(w, grid + i, sizeof(w));
    if ((w[0] | w[1] | w[2] | w[3] | w[4] | w[5] | w[6] | w[7]) & mask) return true;
  }
  for (; i < n; i++) if (grid[i] & ILF_BI_INTRA) return true;
  return false;
}

// Grids cover the rows the context holds (units_h = held rows / 4); ctu_slice covers the full picture.
int ilf_set_deblock_info(ilf_ctx* ctx, int slot, const ilf_deblock_params* params, const uint32_t* info, const uint32_t* info_chroma,
                         const int16_t* mv16, const int32_t* mv32, const uint8_t* ctu_slice) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!params || !info) return fail(ctx, ILF_ERR_ARG, "null params/info");
  if (mv16 && mv32) return fail(ctx, ILF_ERR_ARG, "give mv16 or mv32, not both");
  if (params->num_slices < 1 || params->num_slices > ILF_MAX_SLICES) return fail(ctx, ILF_ERR_ARG, "num_slices %d out of range", params->num_slices);
  Slot& s = ctx->slots[slot];
  size_t cur;
  if (int rc = side_begin(ctx, s, 0, cur)) return rc;
  if (int rc = stage_side(ctx, s, 0, s.db_params, params, sizeof(*params), cur)) return rc;
  if (int rc = stage_grid(ctx, s, s.info, info, 4, cur)) return rc;
  s.has_ctree = info_chroma != nullptr;
  if (info_chroma) if (int rc = stage_grid(ctx, s, s.info_c, info_chroma, 4, cur)) return rc;
  s.mv_mode = mv16 ? 1 : (mv32 ? 2 : 0);
  if (mv16) if (int rc = stage_grid(ctx, s, s.mv, mv16, 8, cur)) return rc;
  if (mv32) if (int rc = stage_grid(ctx, s, s.mv, mv32, 16, cur)) return rc;
  if (ctu_slice) if (int rc = stage_side(ctx, s, 0, s.ctu_slice, ctu_slice, ctx->num_ctus, cur)) return rc;
  s.dev.info = s.info;
  s.dev.info_c = info_chroma ? s.info_c : nullptr;
  s.dev.mv16 = mv16 ? (const int16_t*)s.mv : nullptr;
  s.dev.mv32 = mv32 ? (const int32_t*)s.mv : nullptr;
  s.dev.ctu_slice = ctu_slice ? s.ctu_slice : nullptr;
  s.dev.db_params = s.db_params;
  // The edge records the deblocking kernel reads, derived on s_rec behind the copies just issued (while those arrays are in L2) and
  // behind the slot's previous kernels (side_begin ordered s_up after them); later kernels of the slot wait for ev_rec (join).
  CU(ctx, cudaEventRecord(s.ev_side[0], ctx->s_up));
  CU(ctx, cudaStreamWaitEvent(ctx->s_rec, s.ev_side[0], 0));
  launch_deblock_records(ctx->g, s.db_params, s.info, s.dev.info_c, s.dev.mv16, s.dev.mv32, params->num_slices > 1 ? s.dev.ctu_slice : nullptr, s.db_rec, ctx->s_rec);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaEventRecord(s.ev_rec, ctx->s_rec));
  s.rec_pending = true;
  // A chroma edge is filtered only when a side is intra (bS == 2, LoopFilter.cpp:769): without an intra unit in the layer the
  // chroma decisions read, deblocking leaves both chroma planes as uploaded, and run_stage skips them.
  s.db_chroma = any_intra(info_chroma ? info_chroma : info, (size_t)ctx->g.units_w * ctx->g.units_h);
  s.has_db = true;
  return side_end(ctx, slot, 0);
}

int ilf_set_sao_params(ilf_ctx* ctx, int slot, const ilf_sao_ctu* ctus) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!ctus) return fail(ctx, ILF_ERR_ARG, "null SAO parameters");
  for (int i = 0; i < ctx->num_ctus; i++)
    for (int c = 0; c < 3; c++)
      if (ctus[i].type[c] < ILF_SAO_OFF || ctus[i].type[c] > ILF_SAO_BO) return fail(ctx, ILF_ERR_ARG, "CTU %d comp %d: bad SAO type %d", i, c, ctus[i].type[c]);
  Slot& s = ctx->slots[slot];
  for (int c = 0; c < 3; c++) s.sao_on[c] = false;
  for (int i = 0; i < ctx->num_ctus; i++)
    for (int c = 0; c < 3; c++) {
      if (ctus[i].type[c] == ILF_SAO_OFF) continue;
      s.sao_on[c] = true;
      // offsets are at most 31 << log2OffsetScale with log2OffsetScale <= bitDepth - 10 (SampleAdaptiveOffset.h getMaxOffsetQVal): int8 for <= 12 bit
      for (int k = 0; k < 4; k++)
        if (ctus[i].offset[c][k] < -128 || ctus[i].offset[c][k] > 127)
          return fail(ctx, ILF_ERR_UNSUPPORTED, "CTU %d comp %d: SAO offset %d outside [-128,127]", i, c, ctus[i].offset[c][k]);
    }
  size_t cur;
  if (int rc = side_begin(ctx, s, 1, cur)) return rc;
  if (int rc = stage_side(ctx, s, 1, s.sao, ctus, sizeof(ilf_sao_ctu) * ctx->num_ctus, cur)) return rc;
  s.dev.sao = s.sao;
  s.has_sao = true;
  return side_end(ctx, slot, 1);
}

int ilf_set_alf_params(ilf_ctx* ctx, int slot, const ilf_alf_params* params, const uint8_t* ctu_enable) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!params || !ctu_enable) return fail(ctx, ILF_ERR_ARG, "null ALF parameters");
  Slot& s = ctx->slots[slot];
  for (int c = 0; c < 3; c++) {
    s.alf_on[c] = false;
    for (int i = 0; i < ctx->num_ctus; i++) s.alf_on[c] |= ctu_enable[(size_t)c * ctx->num_ctus + i] != 0;
  }
  size_t cur;
  if (int rc = side_begin(ctx, s, 2, cur)) return rc;
  if (int rc = stage_side(ctx, s, 2, s.alf, params, sizeof(*params), cur)) return rc;
  if (int rc = stage_side(ctx, s, 2, s.alf_ctu_enable, ctu_enable, 3 * (size_t)ctx->num_ctus, cur)) return rc;
  {
    // Coefficient order after transposition (filterBlk, AdaptiveLoopFilter.cpp:541-575), expanded once per picture so
    // that a 4x4 block fetches its 13 (7) coefficients with four 16-byte loads.
    static const uint8_t perm7[4][13] = {{0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12}, {9, 4, 10, 8, 1, 5, 11, 7, 3, 0, 2, 6, 12},
                                         {0, 3, 2, 1, 8, 7, 6, 5, 4, 9, 10, 11, 12}, {9, 8, 10, 4, 3, 7, 11, 5, 1, 0, 2, 6, 12}};
    static const uint8_t perm5[4][7] = {{0, 1, 2, 3, 4, 5, 6}, {4, 1, 5, 3, 0, 2, 6}, {0, 3, 2, 1, 4, 5, 6}, {4, 3, 5, 1, 0, 2, 6}};
    int tab[25][4][16];
    const bool is7 = params->luma_filter_7x7 != 0;
    for (int cl = 0; cl < 25; cl++)
      for (int tr = 0; tr < 4; tr++)
        for (int k = 0; k < 16; k++)
          tab[cl][tr][k] = is7 ? (k < 13 ? params->luma_coeff[cl][perm7[tr][k]] : 0) : (k < 7 ? params->luma_coeff[cl][perm5[tr][k]] : 0);
    if (int rc = stage_side(ctx, s, 2, s.alf_coef, tab, sizeof(tab), cur)) return rc;
    // The same filters in the dot-product layout (ilf_alf_tab.cuh); a picture whose outer coefficients do not fit int8 keeps
    // the general path.
    uint32_t dp[ALF_DP_WORDS];
    bool luma_ok = true, luma_nhi = false;
    for (int cl = 0; cl < 25 && luma_ok; cl++)
      for (int tr = 0; tr < 4; tr++) {
        uint32_t* e = dp + (cl * 4 + tr) * alftab::LUMA_WORDS;
        luma_ok &= is7 ? alftab::build_entry<3, 3>(tab[cl][tr], e, alftab::LUMA_WORDS, &luma_nhi) : alftab::build_entry<3, 2>(tab[cl][tr], e, alftab::LUMA_WORDS, &luma_nhi);
      }
    // the chroma filter (meaningful only when chroma ALF is on: a slice without it leaves the array unset)
    bool chroma_nhi = false;
    int fc[7];
    for (int k = 0; k < 7; k++) fc[k] = params->chroma_coeff[k];
    const bool chroma_ok = alftab::build_entry<2, 2>(fc, dp + 25 * 4 * alftab::LUMA_WORDS, alftab::CHROMA_WORDS, &chroma_nhi);
    s.dev.alf_mode = (luma_ok ? 1 : 0) | (chroma_ok ? 2 : 0) | (luma_ok && !luma_nhi ? 4 : 0) | (chroma_ok && !chroma_nhi ? 8 : 0);
    s.alf_is7 = is7;
    if (int rc = stage_side(ctx, s, 2, s.alf_coef_dp, dp, sizeof(dp), cur)) return rc;
  }
  s.dev.alf_coef = s.alf_coef;
  s.dev.alf_coef_dp = s.alf_coef_dp;
  s.dev.alf = s.alf;
  s.dev.alf_ctu_enable = s.alf_ctu_enable;
  s.has_alf = true;
  return side_end(ctx, slot, 2);
}

// One stage over a batch of slots on stream `st` (ring: its run ring, which also picks its deblocking tile queue).  Buffer rotation
// per plane: the stage reads the plane's current buffer and writes the other work buffer (1 or 2), never buffer 0, so the uploaded
// input survives and ilf_run can be repeated.  Planes for which the stage is off in the whole picture are skipped and keep their
// buffer.  Only the slots i of [first, first + n) with lane_of[i - first] == lane take part.
static int run_stage(ilf_ctx* ctx, int first, int n, int stage, cudaStream_t st, int ring, const uint8_t* lane_of, int lane) {
  const Geom& g = ctx->g;
  const double plane_bytes[3] = {2.0 * g.width * g.rows * 2, 2.0 * (g.width / 2) * (g.rows / 2) * 2, 2.0 * (g.width / 2) * (g.rows / 2) * 2};  // read + write
  for (int c0 = first; c0 < first + n; c0 += MAX_BATCH) {
    const int cn = std::min(MAX_BATCH, first + n - c0);
    // control words of the slots of this chunk (-1: nothing to do), then one compact launch list per kernel
    int word[MAX_BATCH];
    double bytes_of[MAX_BATCH];
    for (int i = 0; i < cn; i++) {
      Slot& s = ctx->slots[c0 + i];
      unsigned v = buf_word(s);
      bool any = false;
      bytes_of[i] = 0;
      for (int p = 0; p < 3; p++) {
        const bool on = lane_of[c0 + i - first] == lane && (stage == 0 ? (p == 0 || s.db_chroma) : (stage == 1 ? s.sao_on[p] : s.alf_on[p]));
        if (!on) { v |= 1u << (6 + p); continue; }
        any = true;
        bytes_of[i] += plane_bytes[p];
        s.result_buf[p] = s.result_buf[p] == 1 ? 2 : 1;
      }
      if (stage == 2) v |= ((s.dev.alf_mode & 1) ? CTL_ALF_DOT_Y : 0) | (s.alf_is7 ? CTL_ALF_7X7 : 0) | ((s.dev.alf_mode & 4) ? CTL_ALF_HIC_Y : 0) |
                       ((s.dev.alf_mode & 2) ? CTL_ALF_DOT_C : 0) | ((s.dev.alf_mode & 8) ? CTL_ALF_HIC_C : 0);
      word[i] = any ? (int)v : -1;
    }
    // one launch of `kernel_launch` over the active slots
    auto stage_launch = [&](auto kernel_launch) -> int {
      BatchCtl ctl;
      const int m = compact(ctx, c0, cn, -1, ctl, [&](int i) { return word[i]; });
      if (!m) return ILF_OK;
      double bytes = 0;
      for (int j = 0; j < m; j++) bytes += bytes_of[ctl.slot[j]];
      return launch(ctx, stage, bytes, 1, [&] { kernel_launch(ctl, m); });
    };
    if (stage == 0) {
      if (int rc = stage_launch([&](const BatchCtl& ctl, int m) { launch_deblock(g, ctx->slots_dev, c0, m, ctl, ctx->db_work + 2 * ring, st); })) return rc;
    } else if (stage == 1) {
      if (int rc = stage_launch([&](const BatchCtl& ctl, int m) { launch_sao(g, ctx->slots_dev, c0, m, ctl, st); })) return rc;
    } else {
      // luma and chroma bands are CTAs of one launch (they share the SMs), accounted under ILF_KERNEL_ALF_LUMA
      if (int rc = stage_launch([&](const BatchCtl& ctl, int m) { launch_alf(g, ctx->slots_dev, c0, m, ctl, st); })) return rc;
    }
  }
  return ILF_OK;
}

int ilf_run(ilf_ctx* ctx, int first_slot, int num_slots, unsigned stages) {
  if (int rc = check_range(ctx, first_slot, num_slots)) return rc;
  if (!(stages & ILF_STAGE_ALL)) return fail(ctx, ILF_ERR_ARG, "empty stage mask");
  // validate every requested stage of every slot before anything is launched or any buffer rotation is recorded
  for (int i = first_slot; i < first_slot + num_slots; i++) {
    const Slot& s = ctx->slots[i];
    if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: run before upload", i);
    for (int st = 0; st < 3; st++) {
      if (!(stages & (1u << st))) continue;
      const bool have = st == 0 ? s.has_db : (st == 1 ? s.has_sao : s.has_alf);
      if (!have) return fail(ctx, ILF_ERR_STATE, "slot %d: side information of stage %d not set since the last upload", i, st);
    }
  }
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  // A full run always restarts from the uploaded input.
  if (stages & ILF_STAGE_DEBLOCK)
    for (int i = first_slot; i < first_slot + num_slots; i++) ctx->slots[i].result_buf[0] = ctx->slots[i].result_buf[1] = ctx->slots[i].result_buf[2] = 0;
  // A chain over a large batch is dealt to the lanes (groups of slots, each group's stages on its own stream): the groups are
  // independent, so one group's kernel fills the SMs that another group's draining kernel leaves idle.  Slots are dealt by estimated
  // cost (planes x stages that run, ALF counted double), heaviest first to the least loaded lane, so that every lane carries a
  // similar mix of kernels.  Per-kernel timing keeps everything on the compute stream (serial kernels are what it measures).
  const bool chain = (stages & (stages - 1)) != 0;
  const int lanes = (ctx->num_lanes > 1 && chain && !ctx->timing && num_slots >= ctx->lane_min_slots) ? ctx->num_lanes : 1;
  std::vector<uint8_t> lane_of(num_slots, 0);
  if (lanes > 1) {
    std::vector<std::pair<int, int>> cost(num_slots);
    for (int i = 0; i < num_slots; i++) {
      const Slot& s = ctx->slots[first_slot + i];
      int c = 0;
      for (int p = 0; p < 3; p++) {
        const int w = p == 0 ? 4 : 1;
        if ((stages & ILF_STAGE_DEBLOCK) && (p == 0 || s.db_chroma)) c += w;
        if ((stages & ILF_STAGE_SAO) && s.sao_on[p]) c += w;
        if ((stages & ILF_STAGE_ALF) && s.alf_on[p]) c += 2 * w;
      }
      cost[i] = {-c, i};
    }
    std::sort(cost.begin(), cost.end());
    int load[ilf_ctx::MAX_LANES] = {};
    for (auto& ci : cost) {
      int best = 0;
      for (int l = 1; l < lanes; l++) if (load[l] < load[best]) best = l;
      lane_of[ci.second] = (uint8_t)best;
      load[best] -= ci.first;
    }
  }
  int rc = ILF_OK;
  for (int gi = 0; gi < lanes; gi++) {
    const int ring = lanes == 1 ? 0 : 1 + gi;
    cudaStream_t st = lanes == 1 ? ctx->stream : ctx->lane[gi];
    int member = -1;
    for (int i = 0; i < num_slots; i++) {
      if (lane_of[i] != gi) continue;
      member = first_slot + i;
      if (int rc2 = join(ctx, ctx->slots[member], st, true)) return rc2;
    }
    if (member < 0) continue;
    for (int k = 0; k < 3 && rc == ILF_OK; k++)
      if (stages & (1u << k)) rc = run_stage(ctx, first_slot, num_slots, k, st, ring, lane_of.data(), gi);
    // whatever was launched is fenced, also on an error path: later uploads / downloads of these slots wait for it
    if (int rc2 = fence(ctx, first_slot, num_slots, st, ring, lane_of.data(), gi)) return rc2;
    if (lanes > 1) CU(ctx, cudaStreamWaitEvent(ctx->stream, ctx->slots[member].ev_run, 0));   // the compute stream joins the lane (the lane does not wait for anything)
  }
  return rc;
}

int ilf_deblock(ilf_ctx* ctx, int slot) { if (int rc = check_slot(ctx, slot)) return rc; return ilf_run(ctx, slot, 1, ILF_STAGE_DEBLOCK); }
int ilf_sao(ilf_ctx* ctx, int slot) { if (int rc = check_slot(ctx, slot)) return rc; return ilf_run(ctx, slot, 1, ILF_STAGE_SAO); }
int ilf_alf(ilf_ctx* ctx, int slot) { if (int rc = check_slot(ctx, slot)) return rc; return ilf_run(ctx, slot, 1, ILF_STAGE_ALF); }

int ilf_alf_classify(ilf_ctx* ctx, int slot, uint8_t* out) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null output");
  Slot& s = ctx->slots[slot];
  if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: classify before upload", slot);
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = join(ctx, s, ctx->stream, false)) return rc;
  BatchCtl ctl;
  ctl.v[0] = (uint16_t)buf_word(s);
  ctl.slot[0] = 0;
  if (int rc = launch(ctx, -1, 0, 1, [&] { launch_alf_classify(ctx->g, ctx->slots_dev, slot, 1, ctl, ctx->stream); })) return rc;
  CU(ctx, cudaMemcpyAsync(out, s.alf_class, (size_t)ctx->g.units_w * ctx->g.units_h, cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return ILF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Encoder SAO statistics (include/ilf_b200.h; EncSampleAdaptiveOffset::getStatistics)
// ---------------------------------------------------------------------------------------------------------------
// Copies the source picture's LOCAL luma rows [first, first + n) of the held region (chroma rows halved) and the full picture's
// ctu_avail.  The original lives in the held-row layout of the slot's buffers, so the kernels address it as they address the picture.
// The original's buffers (allocated on first use), and the upload stream ordered after the slot's kernels: a statistics kernel of the
// previous picture may still read the planes and ctu_avail.
static int original_begin(ilf_ctx* ctx, Slot& s) {
  if (!s.org) {
    CU(ctx, cudaMalloc(&s.org, ctx->buf_elems * sizeof(int16_t)));
    CU(ctx, cudaMalloc(&s.stats_avail, ctx->num_ctus));
    CU(ctx, cudaMalloc(&s.stats, (size_t)ctx->num_ctus * 3 * ILF_SAO_STATS_WORDS * sizeof(long long)));
    s.dev.org[0] = s.org; s.dev.org[1] = s.org + ctx->plane_y; s.dev.org[2] = s.org + ctx->plane_y + ctx->plane_c;
    s.dev.stats_avail = s.stats_avail;
    s.dev.stats = s.stats;
  }
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, s.ev_run, 0));
  return ILF_OK;
}

// The full picture's ctu_avail from host memory; a pageable array is copied before the call returns (the caller may reuse it).
static int original_avail(ilf_ctx* ctx, Slot& s, const uint8_t* ctu_avail) {
  CU(ctx, cudaMemcpyAsync(s.stats_avail, ctu_avail, ctx->num_ctus, cudaMemcpyHostToDevice, ctx->s_up));
  if (!is_pinned(ctu_avail)) CU(ctx, cudaStreamSynchronize(ctx->s_up));
  return ILF_OK;
}

// After the original's copies are issued: the statistics and the search of the slot may run.
static int original_end(ilf_ctx* ctx, int slot) {
  Slot& s = ctx->slots[slot];
  s.has_org = true;
  s.org_since_upload = true;
  return push_desc(ctx, slot);
}

// A whole-picture context takes the original at any time; a band context after the slot's upload (ilf_set_original_band).
static int check_original(ilf_ctx* ctx, int slot, bool band_call) {
  if (ctx->is_band != band_call)
    return fail(ctx, ILF_ERR_STATE, band_call ? "not a band context (ilf_set_original takes the whole picture)" : "SAO statistics are not available on band contexts");
  if (band_call && !ctx->slots[slot].uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: ilf_set_original_band before the slot's upload", slot);
  return ILF_OK;
}

static int set_original_rows(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr,
                             const uint8_t* ctu_avail, int first, int n) {
  if (!y || !cb || !cr || !ctu_avail) return fail(ctx, ILF_ERR_ARG, "null pointer");
  cudaMemoryType types[3];
  if (int rc = refuse_device_planes(ctx, y, cb, cr, types, "ilf_set_original_device")) return rc;
  Slot& s = ctx->slots[slot];
  const Geom& g = ctx->g;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = original_begin(ctx, s)) return rc;
  const int16_t* srcs[3] = {y, cb, cr};
  const ptrdiff_t strides[3] = {sy, scb, scr};
  for (int p = 0; p < 3; p++) {
    const PlaneRows pr = plane_rows(g, p, first, n);
    // pageable sources are staged by the runtime (the call returns when the source may be reused); page-locked ones are asynchronous
    CU(ctx, cudaMemcpy2DAsync(const_cast<int16_t*>(s.dev.org[p]) + (size_t)pr.r0 * pr.pitch, (size_t)pr.pitch * 2, srcs[p], (size_t)strides[p] * 2, (size_t)pr.w * 2, pr.h,
                              cudaMemcpyHostToDevice, ctx->s_up));
  }
  if (int rc = original_avail(ctx, s, ctu_avail)) return rc;
  return original_end(ctx, slot);
}

int ilf_set_original(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr, const uint8_t* ctu_avail) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (int rc = check_original(ctx, slot, false)) return rc;
  return set_original_rows(ctx, slot, y, sy, cb, scb, cr, scr, ctu_avail, 0, ctx->g.height);
}

// Host planes cover the band's OWN rows, as for ilf_upload_band; the statistics and the search read the original at own samples only.
int ilf_set_original_band(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t sy, const int16_t* cb, ptrdiff_t scb, const int16_t* cr, ptrdiff_t scr,
                          const uint8_t* ctu_avail) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (int rc = check_original(ctx, slot, true)) return rc;
  return set_original_rows(ctx, slot, y, sy, cb, scb, cr, scr, ctu_avail, ctx->g.out_row0 - ctx->g.row0, ctx->g.out_rows);
}

// ---------------------------------------------------------------------------------------------------------------
// Pictures in device memory (include/ilf_b200.h): one conversion kernel per call (ilf_io.cu) on the upload or download stream,
// bridged to the caller's stream with an event in each direction; the slot's state changes are those of the host calls.
// ---------------------------------------------------------------------------------------------------------------
// The caller's planes and format, validated before anything is enqueued: `depth` receives the caller's luma / chroma depths,
// `bytes` its sample size.
struct DevicePlanes { const void* p[3]; ptrdiff_t stride[3]; int depth[2], bytes; };
static int check_device_planes(ilf_ctx* ctx, DevicePlanes& d, const ilf_samples* fmt) {
  const Geom& g = ctx->g;
  const ilf_samples dflt = {ILF_SAMPLES_I16, {0, 0}};
  if (!fmt) fmt = &dflt;
  if (fmt->type != ILF_SAMPLES_I16 && fmt->type != ILF_SAMPLES_U8) return fail(ctx, ILF_ERR_ARG, "unknown sample type %d", (int)fmt->type);
  const bool i16 = fmt->type == ILF_SAMPLES_I16;
  for (int c = 0; c < 2; c++) {
    const int v = fmt->bit_depth[c];
    if (i16 ? (v != 0 && (v < 8 || v > 16)) : (v != 0 && v != 8))
      return fail(ctx, ILF_ERR_ARG, "%s depth %d outside %s", c ? "chroma" : "luma", v, i16 ? "8..16 (0: the context's)" : "8 (uint8 samples)");
    d.depth[c] = v ? v : (i16 ? (c ? g.bd_chroma : g.bd_luma) : 8);
  }
  d.bytes = i16 ? 2 : 1;
  for (int p = 0; p < 3; p++) {
    if (!d.p[p]) return fail(ctx, ILF_ERR_ARG, "null plane pointer");
    int dev = -1;
    const cudaMemoryType t = mem_type(d.p[p], &dev);
    if (t != cudaMemoryTypeDevice || dev != ctx->cfg.device)
      return fail(ctx, ILF_ERR_ARG, "plane %d is %s, not device memory of the context's device %d", p,
                  t == cudaMemoryTypeDevice ? "memory of another device" : (t == cudaMemoryTypeManaged ? "managed memory" : "host memory"), ctx->cfg.device);
    if (i16 && ((uintptr_t)d.p[p] & 1)) return fail(ctx, ILF_ERR_ARG, "int16 plane %d is not 2-byte aligned", p);
    const int w = p ? g.width / 2 : g.width;
    if (d.stride[p] < w) return fail(ctx, ILF_ERR_ARG, "plane %d: stride %lld shorter than the plane's width %d", p, (long long)d.stride[p], w);
  }
  return ILF_OK;
}

// The copy between the caller's planes and the context's planes `mine` (held-row layout, first row = LOCAL row 0) over the rows a device
// transfer covers: to_ctx = caller -> context (upload, original), else context -> caller (download).
static IoBatch device_batch(const ilf_ctx* ctx, const DevicePlanes& d, int16_t* const mine[3], bool to_ctx) {
  const Geom& g = ctx->g;
  const int first = g.out_row0 - g.row0, n = g.out_rows;   // a whole picture, or a band's own rows
  IoBatch b;
  for (int p = 0; p < 3; p++) {
    const PlaneRows pr = plane_rows(g, p, first, n);
    const int c = p ? 1 : 0, ctx_depth = c ? g.bd_chroma : g.bd_luma;
    const int diff = to_ctx ? ctx_depth - d.depth[c] : d.depth[c] - ctx_depth;
    int16_t* rows = mine[p] + (size_t)pr.r0 * pr.pitch;
    const long long caller_pitch = (long long)d.stride[p] * d.bytes, ctx_pitch = (long long)pr.pitch * 2;
    IoPlane& io = b.p[p];
    io.src = to_ctx ? d.p[p] : rows;
    io.dst = to_ctx ? (void*)rows : const_cast<void*>(d.p[p]);
    io.src_pitch = to_ctx ? caller_pitch : ctx_pitch;
    io.dst_pitch = to_ctx ? ctx_pitch : caller_pitch;
    io.w = pr.w; io.h = pr.h;
    io.up = std::max(diff, 0); io.down = std::max(-diff, 0);
    io.maxv = (1 << (to_ctx ? ctx_depth : d.depth[c])) - 1;
  }
  b.src_bytes = to_ctx ? d.bytes : 2;
  b.dst_bytes = to_ctx ? 2 : d.bytes;
  return b;
}

// Records the caller's stream up to this call.  First thing enqueued: a stream the context cannot wait for (another device's) fails
// before anything of the transfer is issued.
static int caller_mark(ilf_ctx* ctx, void* stream) {
  CU(ctx, cudaEventRecord(ctx->ev_caller, (cudaStream_t)stream));
  return ILF_OK;
}

int ilf_upload_device(ilf_ctx* ctx, int slot, const void* y, ptrdiff_t sy, const void* cb, ptrdiff_t scb, const void* cr, ptrdiff_t scr,
                      const ilf_samples* fmt, void* stream) {
  if (int rc = check_slot(ctx, slot)) return rc;
  DevicePlanes d = {{y, cb, cr}, {sy, scb, scr}};
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = check_device_planes(ctx, d, fmt)) return rc;
  Slot& s = ctx->slots[slot];
  int16_t* const mine[3] = {plane_ptr(ctx, s, 0, 0), plane_ptr(ctx, s, 0, 1), plane_ptr(ctx, s, 0, 2)};
  const IoBatch b = device_batch(ctx, d, mine, true);
  if (int rc = caller_mark(ctx, stream)) return rc;
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, ctx->ev_caller, 0));
  if (int rc = upload_begin(ctx, s)) return rc;
  if (int rc = launch(ctx, -1, 0, 1, [&] { launch_io_convert(b, ctx->s_up); })) return rc;
  if (int rc = upload_end(ctx, s)) return rc;
  CU(ctx, cudaStreamWaitEvent((cudaStream_t)stream, s.ev_up, 0));
  return ILF_OK;
}

int ilf_set_original_device(ilf_ctx* ctx, int slot, const void* y, ptrdiff_t sy, const void* cb, ptrdiff_t scb, const void* cr, ptrdiff_t scr,
                            const uint8_t* ctu_avail, const ilf_samples* fmt, void* stream) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!ctu_avail) return fail(ctx, ILF_ERR_ARG, "null pointer");
  if (mem_type(ctu_avail) == cudaMemoryTypeDevice) return fail(ctx, ILF_ERR_ARG, "ctu_avail is device memory: it is read from the host");
  DevicePlanes d = {{y, cb, cr}, {sy, scb, scr}};
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = check_device_planes(ctx, d, fmt)) return rc;
  if (int rc = check_original(ctx, slot, ctx->is_band)) return rc;   // ilf_set_original, or ilf_set_original_band on a band context
  Slot& s = ctx->slots[slot];
  if (int rc = caller_mark(ctx, stream)) return rc;
  if (int rc = original_begin(ctx, s)) return rc;
  // ctu_avail is not ordered after the caller's stream: a pageable array is copied, and waited for, without waiting for the caller's work
  if (int rc = original_avail(ctx, s, ctu_avail)) return rc;
  int16_t* const org[3] = {const_cast<int16_t*>(s.dev.org[0]), const_cast<int16_t*>(s.dev.org[1]), const_cast<int16_t*>(s.dev.org[2])};
  const IoBatch b = device_batch(ctx, d, org, true);
  CU(ctx, cudaStreamWaitEvent(ctx->s_up, ctx->ev_caller, 0));
  if (int rc = launch(ctx, -1, 0, 1, [&] { launch_io_convert(b, ctx->s_up); })) return rc;
  if (int rc = original_end(ctx, slot)) return rc;
  CU(ctx, cudaStreamWaitEvent((cudaStream_t)stream, s.ev_up, 0));
  return ILF_OK;
}

int ilf_download_device(ilf_ctx* ctx, int slot, void* y, ptrdiff_t sy, void* cb, ptrdiff_t scb, void* cr, ptrdiff_t scr, const ilf_samples* fmt,
                        void* stream) {
  if (int rc = check_slot(ctx, slot)) return rc;
  DevicePlanes d = {{y, cb, cr}, {sy, scb, scr}};
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = check_device_planes(ctx, d, fmt)) return rc;
  Slot& s = ctx->slots[slot];
  if (!s.uploaded) return fail(ctx, ILF_ERR_STATE, "slot %d: download before upload", slot);
  // each plane from the buffer its last stage left it in
  int16_t* const cur[3] = {plane_ptr(ctx, s, s.result_buf[0], 0), plane_ptr(ctx, s, s.result_buf[1], 1), plane_ptr(ctx, s, s.result_buf[2], 2)};
  const IoBatch b = device_batch(ctx, d, cur, false);
  if (int rc = caller_mark(ctx, stream)) return rc;
  CU(ctx, cudaStreamWaitEvent(ctx->s_down, ctx->ev_caller, 0));
  if (int rc = download_begin(ctx, s)) return rc;
  if (int rc = launch(ctx, -1, 0, 1, [&] { launch_io_convert(b, ctx->s_down); })) return rc;
  if (int rc = download_end(ctx, s)) return rc;
  CU(ctx, cudaStreamWaitEvent((cudaStream_t)stream, s.ev_down, 0));
  return ILF_OK;
}

// CTUs whose statistics records a slot produces: the picture's, or a band's own (num_ctu_rows x ctus_w).
static int own_ctus(const ilf_ctx* ctx) { return ctx->is_band ? ctx->band.num_ctu_rows * ctx->g.ctus_w : ctx->num_ctus; }

// A band slot is measured only against an original of its own rows given since its upload (ilf_set_original_band).
static bool band_org_missing(const ilf_ctx* ctx, const Slot& s) { return ctx->is_band && !s.org_since_upload; }

int ilf_sao_stats(ilf_ctx* ctx, int first_slot, int num_slots) {
  if (int rc = check_range(ctx, first_slot, num_slots)) return rc;
  for (int i = first_slot; i < first_slot + num_slots; i++) {
    const Slot& s = ctx->slots[i];
    if (!s.uploaded || !s.has_org || band_org_missing(ctx, s)) return fail(ctx, ILF_ERR_STATE, "slot %d: statistics need ilf_upload and ilf_set_original", i);
  }
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  const Geom& g = ctx->g;
  for (int i = first_slot; i < first_slot + num_slots; i++)
    if (int rc = join(ctx, ctx->slots[i], ctx->stream, false)) return rc;
  for (int c0 = first_slot; c0 < first_slot + num_slots; c0 += MAX_BATCH) {
    const int cn = std::min(MAX_BATCH, first_slot + num_slots - c0);
    BatchCtl ctl;
    compact(ctx, c0, cn, -1, ctl, [&](int i) { return (int)buf_word(ctx->slots[c0 + i]); });
    // algorithmic bytes: the deblocked and the original picture (own rows) are read once (2 B x 1.5 samples x 2 pictures per luma pixel)
    if (int rc = launch(ctx, ILF_KERNEL_SAO_STATS, 6.0 * g.width * g.out_rows * cn, 1, [&] { launch_sao_stats(g, ctx->slots_dev, c0, cn, ctl, ctx->stream); })) return rc;
  }
  return fence(ctx, first_slot, num_slots, ctx->stream, 0);
}

int ilf_get_sao_stats(ilf_ctx* ctx, int slot, int64_t* out) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null output");
  Slot& s = ctx->slots[slot];
  if (!s.stats) return fail(ctx, ILF_ERR_STATE, "slot %d: no statistics (ilf_set_original / ilf_sao_stats first)", slot);
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  CU(ctx, cudaMemcpyAsync(out, s.stats, (size_t)own_ctus(ctx) * 3 * ILF_SAO_STATS_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return ILF_OK;
}

// Encoder ALF statistics: block classification of the slots' current pictures, then the covariance launches (ilf_alf_stats.cu).
int ilf_alf_stats(ilf_ctx* ctx, int first_slot, int num_slots) {
  if (int rc = check_range(ctx, first_slot, num_slots)) return rc;
  for (int i = first_slot; i < first_slot + num_slots; i++)
    if (band_org_missing(ctx, ctx->slots[i])) return fail(ctx, ILF_ERR_STATE, "not available on band contexts");
  for (int i = first_slot; i < first_slot + num_slots; i++) {
    const Slot& s = ctx->slots[i];
    if (!s.uploaded || !s.has_org) return fail(ctx, ILF_ERR_STATE, "slot %d: statistics need ilf_upload and ilf_set_original", i);
  }
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  const Geom& g = ctx->g;
  const size_t bytes = (size_t)own_ctus(ctx) * ILF_ALF_STATS_WORDS * sizeof(long long);
  for (int i = first_slot; i < first_slot + num_slots; i++) {
    Slot& s = ctx->slots[i];
    if (!s.alf_stats) {
      CU(ctx, cudaMalloc(&s.alf_stats, bytes));
      s.dev.alf_stats = s.alf_stats;
      if (int rc = push_desc(ctx, i)) return rc;
    }
    if (int rc = join(ctx, s, ctx->stream, false)) return rc;
    CU(ctx, cudaMemsetAsync(s.alf_stats, 0, bytes, ctx->stream));
  }
  for (int c0 = first_slot; c0 < first_slot + num_slots; c0 += MAX_BATCH) {
    const int cn = std::min(MAX_BATCH, first_slot + num_slots - c0);
    BatchCtl ctl;
    compact(ctx, c0, cn, -1, ctl, [&](int i) { return (int)buf_word(ctx->slots[c0 + i]); });
    // algorithmic bytes: the reconstructed and the original picture (own rows) are read once (2 B x 1.5 samples x 2 pictures per luma pixel)
    if (int rc = launch(ctx, ILF_KERNEL_ALF_STATS, 6.0 * g.width * g.out_rows * cn, 4, [&] {
          launch_alf_classify(g, ctx->slots_dev, c0, cn, ctl, ctx->stream);
          launch_alf_stats(g, ctx->slots_dev, c0, cn, ctl, ctx->stream);
        }))
      return rc;
  }
  return fence(ctx, first_slot, num_slots, ctx->stream, 0);
}

int ilf_get_alf_stats(ilf_ctx* ctx, int slot, int64_t* out) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null output");
  Slot& s = ctx->slots[slot];
  if (!s.alf_stats) return fail(ctx, ILF_ERR_STATE, "slot %d: no statistics (ilf_set_original / ilf_alf_stats first)", slot);
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  CU(ctx, cudaMemcpyAsync(out, s.alf_stats, (size_t)own_ctus(ctx) * ILF_ALF_STATS_WORDS * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return ILF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Encoder deblocking parameter search (include/ilf_b200.h; EncGOP::applyDeblockingFilterParameterSelection)
// ---------------------------------------------------------------------------------------------------------------
int ilf_deblock_search(ilf_ctx* ctx, int first_slot, int num_slots, const ilf_deblock_candidate* cands, int num_cands, const int32_t shift[2]) {
  if (int rc = check_range(ctx, first_slot, num_slots)) return rc;
  if (!cands || !shift) return fail(ctx, ILF_ERR_ARG, "null pointer");
  if (num_cands < 1 || num_cands > ILF_DEBLOCK_SEARCH_MAX) return fail(ctx, ILF_ERR_ARG, "num_cands %d outside 1..%d", num_cands, ILF_DEBLOCK_SEARCH_MAX);
  if (shift[0] < 0 || shift[0] > 31 || shift[1] < 0 || shift[1] > 31) return fail(ctx, ILF_ERR_ARG, "shift (%d, %d) outside 0..31", shift[0], shift[1]);
  for (int i = first_slot; i < first_slot + num_slots; i++)
    if (band_org_missing(ctx, ctx->slots[i])) return fail(ctx, ILF_ERR_STATE, "not available on band contexts");
  for (int i = first_slot; i < first_slot + num_slots; i++) {
    const Slot& s = ctx->slots[i];
    if (!s.uploaded || !s.has_db || !s.org_since_upload)
      return fail(ctx, ILF_ERR_STATE, "slot %d: the search needs ilf_upload, then ilf_set_deblock_info and ilf_set_original", i);
  }
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  constexpr size_t ROW = (size_t)ILF_DEBLOCK_SEARCH_MAX * 3;
  if (!ctx->search_out) CU(ctx, cudaMalloc(&ctx->search_out, ctx->slots.size() * ROW * sizeof(unsigned long long)));
  for (int i = first_slot; i < first_slot + num_slots; i++)
    if (int rc = join(ctx, ctx->slots[i], ctx->stream, false)) return rc;
  CU(ctx, cudaMemsetAsync(ctx->search_out + first_slot * ROW, 0, num_slots * ROW * sizeof(unsigned long long), ctx->stream));
  for (int c0 = first_slot; c0 < first_slot + num_slots; c0 += MAX_BATCH) {
    const int cn = std::min(MAX_BATCH, first_slot + num_slots - c0);
    for (int mode = 0; mode < 3; mode++) {
      BatchCtl ctl;
      const int m = compact(ctx, c0, cn, mode, ctl, [](int) { return 0; });   // every plane from buffer 0, the uploaded picture
      if (m)
        if (int rc = launch(ctx, -1, 0, 1, [&] {
              launch_deblock_search(ctx->g, ctx->slots_dev, c0, m, ctl, mode, cands, num_cands, shift[0], shift[1], ctx->search_out, ctx->stream);
            }))
          return rc;
    }
  }
  if (int rc = fence(ctx, first_slot, num_slots, ctx->stream, 0)) return rc;
  for (int i = first_slot; i < first_slot + num_slots; i++) ctx->slots[i].search_k = num_cands;
  return ILF_OK;
}

int ilf_get_deblock_search(ilf_ctx* ctx, int slot, uint64_t* out, int max_cands) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!out) return fail(ctx, ILF_ERR_ARG, "null output");
  const Slot& s = ctx->slots[slot];
  if (!s.search_k) return fail(ctx, ILF_ERR_STATE, "slot %d: no deblocking search yet", slot);
  if (max_cands < s.search_k) return fail(ctx, ILF_ERR_ARG, "max_cands %d < %d candidates of the last search", max_cands, s.search_k);
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  CU(ctx, cudaMemcpyAsync(out, ctx->search_out + (size_t)slot * ILF_DEBLOCK_SEARCH_MAX * 3, (size_t)s.search_k * 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(ctx, cudaStreamSynchronize(ctx->stream));
  return s.search_k;
}

int ilf_set_timing(ilf_ctx* ctx, int enable) {
  if (!ctx) return ILF_ERR_ARG;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = timed_collect(ctx)) return rc;
  if (enable) for (int i = 0; i < ILF_NUM_KERNELS; i++) { ctx->kernel_ms[i] = 0; ctx->kernel_launches[i] = 0; ctx->kernel_bytes[i] = 0; }
  ctx->timing = enable != 0;
  return ILF_OK;
}
int ilf_kernel_times(ilf_ctx* ctx, double ms_sum[ILF_NUM_KERNELS], long long launches[ILF_NUM_KERNELS], double algo_bytes[ILF_NUM_KERNELS]) {
  if (!ctx || !ms_sum || !launches || !algo_bytes) return ILF_ERR_ARG;
  CU(ctx, cudaSetDevice(ctx->cfg.device));
  if (int rc = timed_collect(ctx)) return rc;
  for (int i = 0; i < ILF_NUM_KERNELS; i++) { ms_sum[i] = ctx->kernel_ms[i]; launches[i] = ctx->kernel_launches[i]; algo_bytes[i] = ctx->kernel_bytes[i]; }
  return ILF_OK;
}
long long ilf_launch_count(const ilf_ctx* ctx) { return ctx ? ctx->launches : 0; }
int ilf_run_lanes(const ilf_ctx* ctx) { return ctx ? ctx->num_lanes : ILF_ERR_ARG; }
int ilf_alf_path(ilf_ctx* ctx, int slot) {
  if (int rc = check_slot(ctx, slot)) return rc;
  if (!ctx->slots[slot].has_alf) return fail(ctx, ILF_ERR_STATE, "slot %d: ALF parameters not set", slot);
  return ctx->slots[slot].dev.alf_mode & 3;
}

int ilf_slot_input_planes(ilf_ctx* ctx, int slot, void* planes[3], int32_t pitch[3]) {
  if (int rc = check_slot(ctx, slot)) return rc;
  Slot& s = ctx->slots[slot];
  for (int p = 0; p < 3; p++) { planes[p] = plane_ptr(ctx, s, 0, p); pitch[p] = p ? ctx->g.pitch_c : ctx->g.pitch_y; }
  s.uploaded = true;  // the caller fills the planes on the device
  s.org_since_upload = false;
  s.result_buf[0] = s.result_buf[1] = s.result_buf[2] = 0;
  return ILF_OK;
}

int ilf_slot_output_planes(ilf_ctx* ctx, int slot, void* planes[3], int32_t pitch[3]) {
  if (int rc = check_slot(ctx, slot)) return rc;
  Slot& s = ctx->slots[slot];
  for (int p = 0; p < 3; p++) { planes[p] = plane_ptr(ctx, s, s.result_buf[p], p); pitch[p] = p ? ctx->g.pitch_c : ctx->g.pitch_y; }
  return ILF_OK;
}

void* ilf_stream(ilf_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

}  // extern "C"
