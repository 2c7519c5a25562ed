/*
 * ilf_b200.h -- C ABI of the B200 in-loop filter library (libilf_b200.so).
 *
 * The library owns device-resident picture planes (int16 Pel, 4:2:0) and runs VTM 2.1's
 * picture-level in-loop filter chain on them with hand-written sm_100a kernels:
 *
 *   deblocking   replaces LoopFilter::loopFilterPic              (source/Lib/CommonLib/LoopFilter.cpp:149-230)
 *   SAO          replaces SampleAdaptiveOffset::SAOProcess       (source/Lib/CommonLib/SampleAdaptiveOffset.cpp:564-612)
 *   ALF          replaces AdaptiveLoopFilter::ALFProcess         (source/Lib/CommonLib/AdaptiveLoopFilter.cpp:68-139)
 *
 * The reference has no FFI/plugin interface for this path; its boundary is the public API of those
 * three C++ classes (LoopFilter.h:88-112, SampleAdaptiveOffset.h:66-72, AdaptiveLoopFilter.h:70-117),
 * called once per picture from DecLib::executeLoopFilters (source/Lib/DecoderLib/DecLib.cpp:506-533)
 * and EncGOP::compressGOP (source/Lib/EncoderLib/EncGOP.cpp:2099-2160).  The host shim under
 * vvcsoftware_vtm_b200/shim/ keeps those class interfaces and calls the entry points below; see
 * INTEGRATION.md.  Plain C types only: no C++ objects, no exceptions, no torch types.  Every call
 * returns ILF_OK (0) or a negative ilf_status; ilf_last_error() gives the message.  There is NO CPU
 * fallback: without a CUDA device ilf_create fails with ILF_ERR_CUDA.
 *
 * Threading: calls on one context are serialised by the caller (the reference is single-threaded,
 * SURVEY.md 8b); distinct contexts are independent (one per decoder instance / stream / GPU).
 */
#ifndef ILF_B200_H
#define ILF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ILF_ABI_VERSION 1

typedef enum {
  ILF_OK = 0,
  ILF_ERR_ARG = -1,      /* bad argument (geometry, NULL pointer, slot out of range, ...)          */
  ILF_ERR_CUDA = -2,     /* CUDA runtime error or no usable device                                  */
  ILF_ERR_STATE = -3,    /* call order violated (e.g. run before upload / before side info was set) */
  ILF_ERR_NOMEM = -4,
  ILF_ERR_UNSUPPORTED = -5 /* feature outside the reference configuration (non-4:2:0, PCM restore ..) */
} ilf_status;

typedef struct ilf_ctx ilf_ctx;

/* Stage mask for ilf_run. Order of execution is fixed: deblock -> SAO -> ALF (DecLib.cpp:516-530). */
#define ILF_STAGE_DEBLOCK 1u
#define ILF_STAGE_SAO 2u
#define ILF_STAGE_ALF 4u
#define ILF_STAGE_ALL 7u

/* ---------------------------------------------------------------------------------------------
 * Context = one CUDA device + `num_slots` resident pictures of one geometry.
 * A slot holds the picture's three int16 planes (input + two work buffers), its side information
 * and a pinned host staging buffer.  Mirrors the create()/destroy() pair of the three classes
 * (LoopFilter.cpp:124-142, SampleAdaptiveOffset.cpp:126-145, AdaptiveLoopFilter.cpp:196-272):
 * the decoder re-creates the filters for every picture (DecLib.cpp:747-748,789), so the shim
 * creates ONE context per geometry and re-uses it.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t width;            /* luma width  in samples, multiple of 8 (EncAppCfg.cpp:2297)            */
  int32_t height;           /* luma height in samples, multiple of 8                                 */
  int32_t bit_depth_luma;   /* 8..12 (internal bit depth, SPS::getBitDepth(CHANNEL_TYPE_LUMA))       */
  int32_t bit_depth_chroma; /* 8..12                                                                 */
  int32_t ctu_log2;         /* log2 of CTU size: 5, 6 or 7 (cfg CTUSize 128 -> 7)                    */
  int32_t chroma_format;    /* 1 = 4:2:0 (only value supported, as in every reference cfg)           */
  int32_t device;           /* CUDA device ordinal                                                   */
  int32_t num_slots;        /* resident pictures (>= 1)                                              */
} ilf_config;

int ilf_abi_version(void);
int ilf_create(ilf_ctx** out, const ilf_config* cfg);
int ilf_destroy(ilf_ctx* ctx);
const char* ilf_last_error(const ilf_ctx* ctx); /* ctx may be NULL: last error of failed ilf_create */
int ilf_get_config(const ilf_ctx* ctx, ilf_config* out);

/* ---------------------------------------------------------------------------------------------
 * Picture transfer.  Host planes are int16 (Pel, TypeDef.h:370) with strides in SAMPLES, as a
 * PelBuf gives them (Buffer.h:79-110).  Copies go through the slot's pinned staging buffer and
 * are asynchronous on the context's stream; ilf_sync waits.
 * ilf_upload replaces "the filters read cs.getRecoBuf()"; ilf_download replaces "output is written
 * in place into cs.getRecoBuf()" (LoopFilter.cpp:548, SampleAdaptiveOffset.cpp:586, AdaptiveLoopFilter.cpp:89).
 * ------------------------------------------------------------------------------------------- */
int ilf_upload(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t stride_y, const int16_t* cb,
               ptrdiff_t stride_cb, const int16_t* cr, ptrdiff_t stride_cr);
int ilf_download(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t stride_y, int16_t* cb,
                 ptrdiff_t stride_cb, int16_t* cr, ptrdiff_t stride_cr);
int ilf_sync(ilf_ctx* ctx);
/* Transfer pipeline.  A context has an upload, a compute and a download stream, ordered per slot by events: with
 * several slots in rotation the upload of picture n+1, the kernels of picture n and the download of picture n-1
 * overlap.  When the host planes are page-locked (ilf_host_alloc, ilf_host_register, cudaHostAlloc ...) ilf_upload and
 * ilf_download_async copy straight from / into them and return without waiting; pageable planes are staged through the
 * slot's pinned buffer (ilf_upload copies synchronously into it, ilf_download_async blocks).  ilf_wait(slot) returns
 * when the slot's last download has landed; ilf_download = ilf_download_async + ilf_wait.  Page-locked arrays (planes,
 * and side-information arrays of 4 KiB or more) are read asynchronously: leave them unchanged until the slot's next
 * ilf_run has been followed by ilf_wait / ilf_sync. */
int ilf_download_async(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t stride_y, int16_t* cb,
                       ptrdiff_t stride_cb, int16_t* cr, ptrdiff_t stride_cr);
int ilf_wait(ilf_ctx* ctx, int slot);
void* ilf_host_alloc(size_t bytes);             /* page-locked host memory (NULL on failure) */
void ilf_host_free(void* p);
int ilf_host_register(void* p, size_t bytes);   /* page-lock an existing allocation, e.g. a PelStorage of the DPB */
int ilf_host_unregister(void* p);

/* ---------------------------------------------------------------------------------------------
 * Pictures in device memory.  A caller whose picture is already on the GPU (a GPU decoder's reconstruction, an encoder's source
 * frames, a GPU consumer of the filtered picture) hands its planes over without a trip through host memory.  The planes are
 * plain device memory (cudaMalloc, a torch CUDA tensor, ...) of the context's device: managed memory, host memory and memory of
 * another device are refused.  Strides are in SAMPLES.  On a whole-picture context a call covers the whole picture; on a band
 * context the band's OWN rows (ilf_get_band_rows), as ilf_upload_band / ilf_download_band / ilf_set_original_band do -- the halo
 * rows still come from ilf_band_exchange.
 *
 *   ilf_upload_device        as ilf_upload: side information must be set again, every plane's current picture is the upload
 *   ilf_set_original_device  as ilf_set_original, or on a band context as ilf_set_original_band (ILF_ERR_STATE before the slot's
 *                            upload); ctu_avail is HOST memory, read as ilf_set_original reads it (a pageable array is copied before
 *                            the call returns)
 *   ilf_download_device      writes what ilf_download returns (each plane from the buffer its last stage left it in); ILF_ERR_STATE
 *                            before an upload
 *
 * Samples (fmt, NULL = int16 at the context's depths).  The conversion is per plane: b = the context's depth of the plane's channel,
 * c = the caller's; upload and original go c -> b, download b -> c.  With d = destination depth - source depth, computed in int32
 * and stored as the destination type:
 *   d > 0   v << d                                               (no clipping)
 *   d < 0   clip3(0, 2^dst_depth - 1, (v + (1 << (-d - 1))) >> -d)
 *   d = 0   v, bit for bit: int16 at the context's depth is exactly what ilf_upload / ilf_download move
 * An int16 container holds an unsigned sample (so a 16-bit sample of 65535 is the int16 -1).  This is the scaling of VTM's YUV
 * reader and writer: 8-bit frames for a 10-bit context are shifted left by 2, a 10-bit picture downloaded as uint8 is rounded and
 * clipped.
 *
 * Ordering.  The call returns without waiting.  The transfer runs after all work issued to `stream` before the call and before all
 * work issued to `stream` after it, so the caller may overwrite its source, or read its destination, on `stream` at once.  Inside
 * the context the transfer is ordered as its host twin: an upload or original waits for the slot's last run and download, a
 * download for the slot's last run and upload, and the slot's next run or upload waits for the download.  ilf_wait(slot) and
 * ilf_sync cover these transfers.  `stream` is a cudaStream_t on the context's device (NULL: the legacy default stream).
 *
 * Errors.  ILF_ERR_ARG, before anything is enqueued (the slot is left as it was), for: a NULL pointer, a slot out of range, a plane
 * that is not device memory of the context's device, a stride shorter than the plane's width, an int16 plane that is not 2-byte
 * aligned, an unknown type, a depth outside the ranges below.  The host calls (ilf_upload, ilf_download_async, ilf_set_original
 * and their band twins) return ILF_ERR_ARG for device memory.
 * ------------------------------------------------------------------------------------------- */
#define ILF_SAMPLES_I16 0   /* int16, as every host transfer takes it */
#define ILF_SAMPLES_U8 1    /* one byte per sample                    */
typedef struct {
  int32_t type;          /* ILF_SAMPLES_*                                                                     */
  int32_t bit_depth[2];  /* luma, chroma depth of the CALLER's samples.  I16: 8..16, 0 = the context's; U8: 8 (0 means 8) */
} ilf_samples;

int ilf_upload_device(ilf_ctx* ctx, int slot, const void* y, ptrdiff_t stride_y, const void* cb, ptrdiff_t stride_cb, const void* cr,
                      ptrdiff_t stride_cr, const ilf_samples* fmt, void* stream);
int ilf_download_device(ilf_ctx* ctx, int slot, void* y, ptrdiff_t stride_y, void* cb, ptrdiff_t stride_cb, void* cr, ptrdiff_t stride_cr,
                        const ilf_samples* fmt, void* stream);
int ilf_set_original_device(ilf_ctx* ctx, int slot, const void* y, ptrdiff_t stride_y, const void* cb, ptrdiff_t stride_cb, const void* cr,
                            ptrdiff_t stride_cr, const uint8_t* ctu_avail /* HOST, [ctus_h*ctus_w] */, const ilf_samples* fmt, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Deblocking side information: the packed per-4x4 CU/TU metadata grid.
 *
 * One uint32 per 4x4 luma unit, raster order, units_w = width/4 (what the reference looks up per
 * 4x4 part through CodingStructure::getCU/getTU/getMotionInfo, LoopFilter.cpp:419-541):
 *   bit 0      ILF_BI_INTRA    CU at this unit is MODE_INTRA                         (:433)
 *   bit 1      ILF_BI_CBF      luma cbf of the TU covering the unit, TU::getCbf       (:444)
 *   bit 2      ILF_BI_EDGE_V   the unit's LEFT border is an edge the reference filters: the unit lies
 *                              in a column xDeblockCU walks (edge 0 of a CU whose x is a multiple of 8,
 *                              or an x offset that is a multiple of 64 inside a wider CU, :313-354)
 *                              AND m_aapbEdgeFilter is set there (:372-417)
 *   bit 3      ILF_BI_TU_V     value left in m_aapucBS before bS derivation ("is a TU edge", :386-390,:444)
 *   bit 4,5    ILF_BI_EDGE_H / ILF_BI_TU_H   same for the unit's TOP border
 *   bit 6      ILF_BI_NOFILT   samples of this CU are restored after filtering (ipcm with
 *                              pcm-loop-filter-disable, or transquant bypass; :651-663,:903-915)
 *   bit 7      ILF_BI_BSLICE   the unit's slice is a B slice (:454)
 *   bits 8-15  qp              CodingUnit::qp as int8 (:626)
 *   bits 16-23 ref0            dense id of Slice::getRefPic(L0, refIdx[0]) -- identity of the
 *   bits 24-31 ref1            reference PICTURE, not the index (:456-459); 0xFF = list unused
 * mv: four components per unit {mv0.hor, mv0.ver, mv1.hor, mv1.ver}, zero where the list is unused,
 * all promoted to 1/16 pel when the SPS uses high-precision MVs (Mv::setHighPrec, :468-477); the
 * threshold that goes with them is ilf_deblock_params.mv_threshold (4, or 16 with high precision).
 * They may be given as int16 (mv16) when every component fits, else as int32 (mv32); exactly one
 * of the two pointers is non-NULL (both NULL is allowed for an all-intra picture).
 * info_chroma is the second layer for the separate chroma tree of dual-tree I slices (cu.chType ==
 * CH_C, :182-191): same layout, qp/flags of the chroma-tree CU; NULL when the picture has no
 * dual-tree slice, and then chroma edges are derived from `info` (bS == 2 on the 16-luma-sample grid).
 * ------------------------------------------------------------------------------------------- */
#define ILF_BI_INTRA 0x01u
#define ILF_BI_CBF 0x02u
#define ILF_BI_EDGE_V 0x04u
#define ILF_BI_TU_V 0x08u
#define ILF_BI_EDGE_H 0x10u
#define ILF_BI_TU_H 0x20u
#define ILF_BI_NOFILT 0x40u
#define ILF_BI_BSLICE 0x80u
#define ILF_REF_NONE 0xFFu
#define ILF_MAX_SLICES 64

typedef struct {
  int8_t beta_offset_div2; /* Slice::getDeblockingFilterBetaOffsetDiv2 (:568) */
  int8_t tc_offset_div2;   /* Slice::getDeblockingFilterTcOffsetDiv2   (:569) */
  int8_t reserved[2];
} ilf_slice_params;

typedef struct {
  int32_t cb_qp_offset; /* PPS::getQpOffset(COMPONENT_Cb) (:808) */
  int32_t cr_qp_offset;
  int32_t mv_threshold; /* 4, or 16 when MVs are stored in 1/16 pel (:468-477) */
  int32_t num_slices;   /* entries used in `slices` (1..ILF_MAX_SLICES) */
  ilf_slice_params slices[ILF_MAX_SLICES];
} ilf_deblock_params;

/* ctu_slice: slice index per CTU (raster), NULL = every CTU in slice 0. */
int ilf_set_deblock_info(ilf_ctx* ctx, int slot, const ilf_deblock_params* params,
                         const uint32_t* info, const uint32_t* info_chroma, const int16_t* mv16,
                         const int32_t* mv32, const uint8_t* ctu_slice);

/* ---------------------------------------------------------------------------------------------
 * SAO side information: parameters per CTU and component AFTER merge resolution and offset scaling
 * (xReconstructBlkSAOParams stays on the host, SampleAdaptiveOffset.cpp:265-289, :147-170), plus the
 * eight neighbour-CTU availability flags of deriveLoopFilterBoundaryAvailibility (:685-760).
 * ------------------------------------------------------------------------------------------- */
#define ILF_SAO_OFF (-1)
#define ILF_SAO_EO_0 0
#define ILF_SAO_EO_90 1
#define ILF_SAO_EO_135 2
#define ILF_SAO_EO_45 3
#define ILF_SAO_BO 4

#define ILF_AVAIL_L 0x01u
#define ILF_AVAIL_R 0x02u
#define ILF_AVAIL_A 0x04u
#define ILF_AVAIL_B 0x08u
#define ILF_AVAIL_AL 0x10u
#define ILF_AVAIL_AR 0x20u
#define ILF_AVAIL_BL 0x40u
#define ILF_AVAIL_BR 0x80u

typedef struct {
  int16_t offset[3][4]; /* EO: offsets of edge classes {0,1,3,4} (class 2 is 0, :167);
                           BO: offsets of bands band_pos+0..3 (mod 32), already << log2OffsetScale */
  int8_t type[3];       /* ILF_SAO_OFF or SAOModeNewTypes (TypeDef.h:738-750) per component         */
  uint8_t band_pos[3];  /* BO: typeAuxInfo = first band                                             */
  uint8_t avail;        /* ILF_AVAIL_* of the CTU (derived at the luma position, shared by chroma)  */
  uint8_t reserved;
} ilf_sao_ctu; /* 32 bytes */

int ilf_set_sao_params(ilf_ctx* ctx, int slot, const ilf_sao_ctu* ctus /* [ctus_h*ctus_w] */);

/* ---------------------------------------------------------------------------------------------
 * ALF side information: final coefficients per class (m_coeffFinal after reconstructCoeff,
 * AdaptiveLoopFilter.cpp:141-194, kept on the host), chroma coefficients, luma filter shape and
 * the per-CTU enable flags (Picture::getAlfCtuEnableFlag, Picture.h:309-320).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int16_t luma_coeff[25][13]; /* [classIdx][coef]; 5x5 shape uses the first 7 of each row          */
  int16_t chroma_coeff[7];
  int16_t luma_filter_7x7;    /* 1 = ALF_FILTER_7, 0 = ALF_FILTER_5 (TypeDef.h:1430-1435)          */
} ilf_alf_params;

/* ctu_enable: [3][num_ctus] bytes, component-major. */
int ilf_set_alf_params(ilf_ctx* ctx, int slot, const ilf_alf_params* params,
                       const uint8_t* ctu_enable);

/* ---------------------------------------------------------------------------------------------
 * Execution.  ilf_run launches the requested stages for slots [first_slot, first_slot+num_slots)
 * as one batched launch per stage (pictures of a batch are independent).  A stage in the mask
 * whose side information was not set since the last upload is an error.  The result of a slot is
 * what ilf_download returns; the uploaded input is preserved, so ilf_run can be repeated.
 * Every requested stage of every slot is validated before anything is launched.  The slots of a batch may mix the motion-vector
 * representations (none / mv16 / mv32) and grids with or without a chroma-tree layer: the deblocking stage reads the edge
 * records ilf_set_deblock_info derived and is still one launch (ilf_deblock_search takes one launch per representation present).
 * ilf_deblock / ilf_sao / ilf_alf are the per-class entry points of the shim (one stage, one slot;
 * each consumes the previous stage's output).
 * ------------------------------------------------------------------------------------------- */
int ilf_run(ilf_ctx* ctx, int first_slot, int num_slots, unsigned stages);
int ilf_deblock(ilf_ctx* ctx, int slot);
int ilf_sao(ilf_ctx* ctx, int slot);
int ilf_alf(ilf_ctx* ctx, int slot);

/* ALF block classification of the slot's current picture (AdaptiveLoopFilter::deriveClassification,
 * AdaptiveLoopFilter.cpp:274-463), for parity tests and the encoder (EncAdaptiveLoopFilter.cpp:257):
 * out[units_h][units_w] = classIdx | transposeIdx << 5 per 4x4 luma block. */
int ilf_alf_classify(ilf_ctx* ctx, int slot, uint8_t* out);

/* ---------------------------------------------------------------------------------------------
 * Encoder SAO statistics on the device-resident picture (SURVEY.md 8f): replaces
 * EncSampleAdaptiveOffset::getStatistics (EncoderLib/EncSampleAdaptiveOffset.cpp:278-331, getBlkStats :1122-1487) for the
 * path without SaoCtuBoundary.  ilf_set_original uploads the source picture of the slot (cs.getOrgBuf()) and the per-CTU
 * availability flags (ILF_AVAIL_L / _A / _AL of EncSampleAdaptiveOffset::deriveLoopFilterBoundaryAvailibility; right,
 * below and above-right follow from the picture bounds as in :307-309); ilf_sao_stats launches one kernel over the
 * CURRENT state of the slots' pictures (after ilf_deblock: the deblocked picture, which is what the encoder measures);
 * ilf_get_sao_stats copies a slot's result to the host: out[num_ctus][3][5][64] int64, per CTU, component and SAO type
 * diff[32] followed by count[32] -- the memory layout of SAOStatData (EncSampleAdaptiveOffset.h:53-57).
 * ilf_set_original refuses band contexts; a band context takes its original with ilf_set_original_band (band section below).
 * ------------------------------------------------------------------------------------------- */
#define ILF_SAO_STATS_WORDS (5 * 64)
int ilf_set_original(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t stride_y, const int16_t* cb, ptrdiff_t stride_cb, const int16_t* cr,
                     ptrdiff_t stride_cr, const uint8_t* ctu_avail /* [ctus_h*ctus_w] */);
int ilf_sao_stats(ilf_ctx* ctx, int first_slot, int num_slots);
int ilf_get_sao_stats(ilf_ctx* ctx, int slot, int64_t* out);

/* ---------------------------------------------------------------------------------------------
 * Encoder ALF statistics on the device-resident picture (SURVEY.md 8f): replaces EncAdaptiveLoopFilter::deriveStatsForFiltering /
 * getBlkStats / calcCovariance (EncoderLib/EncAdaptiveLoopFilter.cpp:1317-1514), including the block classification of the picture
 * it measures (deriveClassification, :257).  ilf_alf_stats works on the CURRENT state of the slots' pictures (after ilf_sao: the
 * picture the encoder's ALF search sees) and on the source pictures given with ilf_set_original; ilf_get_alf_stats copies a slot's
 * result to the host: out[num_ctus][ILF_ALF_STATS_WORDS] int64 -- exactly the integers the reference's doubles hold.  Per CTU:
 *   luma  [25 classes][105]   7x7 shape: E[k][l] for k <= l row-major (91), y[k] (13), pixAcc (1)
 *   Cb    [36], Cr [36]       5x5 shape: E (28), y (7), pixAcc
 * The luma statistics of the 5x5 shape (m_filterShapes[CHANNEL_TYPE_LUMA][0]) are rows / columns {2, 5, 6, 7, 10, 11, 12} of the 7x7
 * record: under every transposition the 5x5 taps are those taps of the 7x7 diamond.  On a band context: after ilf_set_original_band.
 * ------------------------------------------------------------------------------------------- */
#define ILF_ALF_STATS_WORDS (25 * 105 + 36 + 36)
int ilf_alf_stats(ilf_ctx* ctx, int first_slot, int num_slots);
int ilf_get_alf_stats(ilf_ctx* ctx, int slot, int64_t* out);

/* ---------------------------------------------------------------------------------------------
 * Encoder deblocking parameter search on the device-resident picture (SURVEY.md 8f): serves
 * EncGOP::applyDeblockingFilterParameterSelection (EncoderLib/EncGOP.cpp:2550-2574, switched on by DeblockingFilterMetric), which
 * deblocks the same reconstruction once per (beta offset, tc offset) candidate and keeps the pair of least distortion
 * (xFindDistortionFrame, :3970).  ilf_deblock_search scores K candidates of every slot in one pass that reads the picture and the
 * original once and writes no picture; ilf_get_deblock_search copies a slot's K x 3 sums to the host:
 *   out[k][c] = sum over the samples of plane c (Y, Cb, Cr) of ((D_k - O)^2 >> shift[c > 0])
 * The shift applies to every sample, as xFindDistortionFrame does; the caller passes the reference's shift
 * (DISTORTION_PRECISION_ADJUSTMENT of its bit depth).  O is the original of ilf_set_original.  D_k is exactly what ilf_deblock
 * produces from the slot's UPLOADED picture with the slot's deblocking side information, the beta_offset_div2 / tc_offset_div2 of
 * EVERY slice replaced by candidate k (the reference sets the same offsets on all slices, :2560-2566); chroma QP offsets,
 * mv_threshold, ctu_slice, grids and motion stay as set.  Offsets are any int8_t; the table index clamps as in deblocking (:626-634).
 * The search reads buffer 0, so stages run since the upload do not change its result, and it writes no picture plane:
 * ilf_download / ilf_run after a search give what they gave before it.
 * Errors: ILF_ERR_ARG for a bad slot range, num_cands outside 1..ILF_DEBLOCK_SEARCH_MAX, NULL pointers or a shift outside 0..31;
 * ILF_ERR_STATE for a slot without an upload, without deblocking side information or without ilf_set_original since its upload,
 * and on a band context without ilf_set_original_band since its upload.  Ordering: the search waits for the slots' uploads and side information, runs on the context's stream and
 * is waited for by the slots' next uploads.  ilf_get_deblock_search synchronises and returns the K of the slot's last search
 * (ILF_ERR_STATE before any search, ILF_ERR_ARG when max_cands < K).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int8_t beta_offset_div2, tc_offset_div2;
} ilf_deblock_candidate;
#define ILF_DEBLOCK_SEARCH_MAX 64
int ilf_deblock_search(ilf_ctx* ctx, int first_slot, int num_slots, const ilf_deblock_candidate* cands, int num_cands,
                       const int32_t shift[2] /* luma, chroma */);
int ilf_get_deblock_search(ilf_ctx* ctx, int slot, uint64_t* out /* [K][3] */, int max_cands);

/* ---------------------------------------------------------------------------------------------
 * Post-filter consumers on the device-resident picture (SURVEY.md 8f): what the decoder does with a picture right after the
 * in-loop filters.
 *   ilf_picture_hash       the two decoded-picture-hash methods that are not inherently serial, calcCRC and calcChecksum
 *                          (source/Lib/CommonLib/PicYuvMD5.cpp:91-175), of the slot's CURRENT picture: out[Y, Cb, Cr] = the 16-bit CRC
 *                          / 32-bit checksum the reference puts into the digest, big-endian, before comparing it with the SEI
 *                          (DecLib.cpp:579-588).  12 bytes come down instead of the picture.  MD5 stays on the host.
 *   ilf_download_extended  ilf_download into planes that have `margin` luma (margin / 2 chroma) samples of room on every side (a
 *                          PelStorage of Picture::create, Picture.cpp:791-…), and the margins filled by replication as
 *                          Picture::extendPicBorder does (Picture.cpp:996-1040) -- the caller marks the picture as extended.
 * Both refuse band contexts: their twins are ilf_picture_hash_band + ilf_hash_combine and ilf_download_band_extended (band section).
 * ------------------------------------------------------------------------------------------- */
#define ILF_HASH_CRC 1
#define ILF_HASH_CHECKSUM 2
int ilf_picture_hash(ilf_ctx* ctx, int slot, int kind, uint32_t out[3]);
int ilf_download_extended(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t stride_y, int16_t* cb, ptrdiff_t stride_cb, int16_t* cr, ptrdiff_t stride_cr,
                          int margin);

/* ---------------------------------------------------------------------------------------------
 * Measurement helpers (bench.py).  Accumulated device time per kernel in milliseconds since
 * ilf_set_timing(ctx, 1) (CUDA event pairs around every launch on the context's stream, collected
 * without synchronising inside ilf_run), number of kernel launches issued since ilf_create (the
 * conversion kernel of the device transfers included; it has no timing slot; the edge-record pass
 * of ilf_set_deblock_info is not counted: the count since ilf_create stays the number of transfer
 * and filter launches, which callers and tests compare against the stages they ran), and raw device
 * pointers of a slot's input planes so that synthetic pictures can be generated on the device.
 * planes[0..2] = Y, Cb, Cr; pitch in samples.  These pointers carry no ordering: a caller's
 * picture enters and leaves through the device transfers above.
 * ------------------------------------------------------------------------------------------- */
#define ILF_KERNEL_DEBLOCK 0
#define ILF_KERNEL_SAO 1
#define ILF_KERNEL_ALF_LUMA 2   /* the whole ALF stage: luma and chroma bands are CTAs of ONE launch */
#define ILF_KERNEL_ALF_CHROMA 3 /* reserved: always zero */
#define ILF_KERNEL_SAO_STATS 4  /* ilf_sao_stats */
#define ILF_KERNEL_ALF_STATS 5  /* ilf_alf_stats: classification + the three statistics launches */
#define ILF_NUM_KERNELS 6
int ilf_set_timing(ilf_ctx* ctx, int enable); /* enable != 0: clear the accumulators and time every launch */
/* algo_bytes: bytes the launches had to move = 2 bytes x (read + write) x samples of the planes they processed
 * (planes whose stage is off for the whole picture are skipped and not counted).  Synchronises the stream. */
int ilf_kernel_times(ilf_ctx* ctx, double ms_sum[ILF_NUM_KERNELS], long long launches[ILF_NUM_KERNELS],
                     double algo_bytes[ILF_NUM_KERNELS]);
long long ilf_launch_count(const ilf_ctx* ctx);
/* Lanes.  ilf_run deals a CHAIN (two or more stages) over a batch of at least ILF_RUN_LANE_MIN slots (default 8) to this many
 * extra compute streams (environment ILF_RUN_LANES at ilf_create, default 2, 1 = off): the slots of a batch are independent
 * pictures, so one lane's kernel fills the SMs that another lane's draining kernel leaves idle, and the instruction-bound ALF
 * CTAs of one lane share SMs with the memory-bound deblocking / SAO CTAs of another.  Every slot still sees its stages in
 * order; the context's stream (ilf_stream) joins the lanes after every run, uploads / downloads / later runs are ordered per
 * slot by events.  Per-kernel timing (ilf_set_timing) keeps a run on the context's stream.  Returns the lane count (1 = off). */
int ilf_run_lanes(const ilf_ctx* ctx);
/* Which arithmetic path the slot's ALF filters take (chosen by ilf_set_alf_params from the coefficient ranges; results are
 * bit-exact either way): bit 0 = luma, bit 1 = chroma on the IDP.2A dot-product path (every coefficient outside the centre and its
 * four neighbours fits int8), else the general 32-bit multiply path.  Negative = ilf_status. */
#define ILF_ALF_PATH_LUMA_DOT 1
#define ILF_ALF_PATH_CHROMA_DOT 2
int ilf_alf_path(ilf_ctx* ctx, int slot);
int ilf_slot_input_planes(ilf_ctx* ctx, int slot, void* planes[3], int32_t pitch[3]);
int ilf_slot_output_planes(ilf_ctx* ctx, int slot, void* planes[3], int32_t pitch[3]);
void* ilf_stream(ilf_ctx* ctx); /* cudaStream_t of the context */

/* ---------------------------------------------------------------------------------------------
 * CTU-row band mode (one picture split across GPUs, BASELINE config 4; SURVEY.md 8e).  A band context is
 * created with the FULL picture geometry plus the band's CTU-row range; it holds the band's own rows and 16
 * luma (8 chroma) halo rows above and below (clipped to the picture; 16 keeps the held region on the chroma edge grid).  The three stages are local stencils:
 * the dependency chain of a band's own rows closes at 4 luma / 3 chroma INPUT rows per side, so the halo
 * is exchanged once per picture, on the input, and every GPU filters its halo rows redundantly.  The
 * results of the halo rows themselves are not valid and are never downloaded.
 *
 *   ilf_upload_band     host planes cover the band's OWN rows only (ilf_get_band_rows: own_first, own_rows)
 *   ilf_band_export     handle of a slot's planes for the neighbouring band contexts
 *   ilf_band_connect    opens a neighbour's planes: direct pointer in the same process (peer access is enabled
 *                       when the devices differ), CUDA IPC mapping from another process (one process per GPU)
 *   ilf_band_exchange   copies the halo rows of the slot's input picture out of the connected neighbours'
 *                       input buffers with one kernel that reads the peer memory directly (NVLink P2P between
 *                       GPUs), on the context's upload stream; the slot's next ilf_run is ordered after it.  The CALLER makes sure that the
 *                       neighbours' uploads have completed (ilf_sync on them; a barrier between processes)
 *                       and that a neighbour does not upload its next picture before this exchange is done.
 *   ilf_download_band   the band's own rows of the filtered picture
 * Side information of a band context: unit grids cover the rows the context HOLDS (ilf_get_band: first_row,
 * num_rows); ctu_slice, SAO parameters and ALF flags cover the full picture.
 *
 * Consumers of the filtered picture on a band context (the band twins of the post-filter and encoder entry points above):
 *   ilf_picture_hash_band  CRC and checksum of the band's OWN rows of the slot's current picture, as a part that ilf_hash_combine
 *                          folds with the other bands' parts into ilf_picture_hash of the whole picture.  crc[p] is what the rows
 *                          contribute to the CRC register from a ZERO register, sum[p] the checksum partial sum (row masks in picture
 *                          coordinates).  The part carries the picture geometry, so parts can travel between processes as bytes.
 *                          Waits for the slot's upload and last run, like ilf_picture_hash, and returns after a synchronise.
 *   ilf_hash_combine       host only, no context: out[Y, Cb, Cr] of ILF_HASH_CRC / ILF_HASH_CHECKSUM from parts in any order.
 *                          ILF_ERR_ARG unless the parts tile [0, height) exactly (no gap, no overlap), share geometry and bit depths,
 *                          num_parts >= 1, kind is valid and no pointer is NULL.
 *   ilf_download_band_extended  ilf_download_band with Picture::extendPicBorder's margins (see ilf_download_extended): the pointers
 *                          address the band's first own row inside the caller's FULL-picture planes, which have `margin` luma
 *                          (margin / 2 chroma) samples of room on every side.  Writes the own rows and their left / right margins,
 *                          the top margin rows (and corners) only when the band owns picture row 0, the bottom ones only when it
 *                          owns the last row; no other row.  Once every band has run into the same planes they equal
 *                          ilf_download_extended of the whole picture.  margin must be even and >= 0.
 *   ilf_set_original_band  the source picture of the band's OWN rows (host planes as ilf_upload_band) and ctu_avail of the FULL
 *                          picture (as ilf_set_original).  After it (since the slot's upload) ilf_sao_stats, ilf_alf_stats,
 *                          ilf_deblock_search and their ilf_get_* accept the band slot:
 *                            statistics records are those of the band's own CTUs, num_ctu_rows x ctus_w records in raster order
 *                            (in band order they concatenate to the whole picture's records); ilf_alf_classify returns the held
 *                            unit rows, whose own rows equal the whole picture's; the search sums cover the own rows (summed over
 *                            the bands they are the whole picture's sums).
 *                          The kernels read the halo rows of the slot's current picture, so the halo must have been exchanged since
 *                          the upload (ilf_band_exchange), as for ilf_run.
 * ilf_picture_hash_band, ilf_download_band_extended and ilf_set_original_band return ILF_ERR_STATE on a whole-picture context
 * and before the slot's upload.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t first_ctu_row; /* first CTU row owned by this band */
  int32_t num_ctu_rows;  /* CTU rows owned                    */
} ilf_band;

typedef struct { unsigned char opaque[192]; } ilf_band_handle;
#define ILF_BAND_ABOVE 0
#define ILF_BAND_BELOW 1

int ilf_create_band(ilf_ctx** out, const ilf_config* cfg, const ilf_band* band);
int ilf_get_band(const ilf_ctx* ctx, ilf_band* out, int32_t* first_row, int32_t* num_rows);
int ilf_get_band_rows(const ilf_ctx* ctx, int32_t* own_first, int32_t* own_rows);
int ilf_upload_band(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t stride_y, const int16_t* cb, ptrdiff_t stride_cb, const int16_t* cr,
                    ptrdiff_t stride_cr);
int ilf_download_band(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t stride_y, int16_t* cb, ptrdiff_t stride_cb, int16_t* cr, ptrdiff_t stride_cr);
int ilf_band_export(ilf_ctx* ctx, int slot, ilf_band_handle* out);
int ilf_band_connect(ilf_ctx* ctx, int slot, int side, const ilf_band_handle* neighbour);
int ilf_band_exchange(ilf_ctx* ctx, int slot);
int ilf_band_exchange_batch(ilf_ctx* ctx, int first_slot, int num_slots); /* the same for several slots with one launch */

typedef struct {
  int32_t width, height, bd_luma, bd_chroma; /* full picture, copied from the context                                   */
  int32_t first_row, num_rows;               /* luma picture rows covered: the band's own rows                          */
  uint32_t crc[3];                           /* per plane: CRC register contribution of these rows from a ZERO register */
  uint32_t sum[3];                           /* per plane: checksum partial sum (mod 2^32), masks in picture coordinates */
} ilf_hash_part;
int ilf_picture_hash_band(ilf_ctx* ctx, int slot, ilf_hash_part* out);
int ilf_hash_combine(const ilf_hash_part* parts, int num_parts, int kind, uint32_t out[3]);
int ilf_download_band_extended(ilf_ctx* ctx, int slot, int16_t* y, ptrdiff_t stride_y, int16_t* cb, ptrdiff_t stride_cb, int16_t* cr,
                               ptrdiff_t stride_cr, int margin);
int ilf_set_original_band(ilf_ctx* ctx, int slot, const int16_t* y, ptrdiff_t stride_y, const int16_t* cb, ptrdiff_t stride_cb, const int16_t* cr,
                          ptrdiff_t stride_cr, const uint8_t* ctu_avail /* [ctus_h*ctus_w], full picture */);

#ifdef __cplusplus
}
#endif
#endif /* ILF_B200_H */
