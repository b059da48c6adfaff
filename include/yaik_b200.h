/* yaik_b200 — C ABI of the B200-native YAIK encoder-analysis stage.
 *
 * The reference (KLab/YAIK) has no plugin/FFI layer: the boundary is four member functions of
 * `struct EncoderContext` called from `EncoderContext::Convert()` plus two global buffers.  Each entry
 * point below names the reference interface it replaces (paths under the reference tree; "EC.cpp" =
 * encoder/EncoderContext.cpp).  The host-side C++ mirror of that class (yaik_b200/host/EncoderContext.h)
 * and the ctypes binding (yaik_b200/capi.py) call nothing but these symbols.
 *
 * Conventions: plain pointers and sizes; every call returns 0 (YK_OK) or a negative YK_ERR_* code; no
 * exceptions cross the boundary; the caller owns every host buffer; a context is used from one thread at
 * a time, distinct contexts are independent (one per GPU / per stream).  There is NO CPU fallback: without
 * a CUDA device every compute entry point fails with YK_ERR_CUDA.
 *
 * Domain (SURVEY.md §8c hazards 7, 11): planes are int32 with samples 0..255 (the reference's
 * `Plane`, encoder/framework.h:74-127, as filled by Image::LoadPNG, Image.cpp:200-229); width and height
 * are multiples of 4 (the reference's loader demands multiples of 8; 4x4 is the last mip level).  A sample
 * outside 0..255 makes the analysis return YK_ERR_RANGE (the reference indexes a 256-bin histogram with it,
 * EC.cpp:8445).  Only the 3-plane RGB form of FittingQuadSmooth (PlaneBit == 7) is provided.
 */
#ifndef YAIK_B200_H
#define YAIK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YK_OK                0
#define YK_ERR_CUDA         -1   /* CUDA runtime error (yk_last_cuda_error() has the text) */
#define YK_ERR_ARG          -2   /* bad argument / size outside the domain */
#define YK_ERR_CAPACITY     -3   /* image or batch larger than the context was created for */
#define YK_ERR_RANGE        -4   /* a sample outside 0..255 was found */
#define YK_ERR_STATE        -5   /* call order: stage not run yet / no image set */
#define YK_ERR_UNSUPPORTED  -6   /* variant of the reference call that this path does not provide */
#define YK_ERR_NOMEM        -7

/* gradient pass ids in the order EncoderContext::Convert() runs them (EC.cpp:9057-9093):
 * (shX,shY) = (4,4) (4,3) (3,4) (3,3) (3,2) (2,3) (2,2)  i.e. 16x16 16x8 8x16 8x8 8x4 4x8 4x4 */
#define YK_NUM_PASSES 7

typedef struct yk_ctx yk_ctx;

int         yk_abi_version(void);
const char* yk_error_string(int code);
const char* yk_last_cuda_error(void);
int         yk_device_count(int* count);

/* One context per GPU (or per stream).  Owns the device planes of `maxSlots` images of up to maxW x maxH
 * (a "slot" holds one image and every result of its analysis; batches are slots 0..n-1 of the same size),
 * the compact state masks, the result streams and pinned staging.  Replaces the EncoderContext
 * constructor/Release pair for this stage (EncoderContext.h:185-232). */
int  yk_create(yk_ctx** out, int device, int maxW, int maxH, int maxPlanes, int maxSlots);
void yk_destroy(yk_ctx* ctx);

/* Work is enqueued on this cudaStream_t (default: a stream the context creates).  Lets a caller time the
 * path with its own CUDA events or order it against its own copies. */
int  yk_set_stream(yk_ctx* ctx, void* cudaStream);
int  yk_sync(yk_ctx* ctx);

/* The analysis kernel is persistent: `ctas` CTAs (0 = one per SM, the default and the best choice for one image at a
 * time).  When independent images are pipelined over several contexts / streams, half the SM count per launch lets two
 * launches run side by side and hides each one's ramp and tail.  yk_sm_count: SMs of the context's device. */
int  yk_set_analysis_ctas(yk_ctx* ctx, int ctas);
int  yk_sm_count(yk_ctx* ctx);

/* Pinned host memory for Plane::pixels so uploads run at full PCIe rate (Plane ctor, framework.h:76). */
void* yk_host_alloc(size_t bytes);
void  yk_host_free(void* p);

/* EncoderContext::SetImageToEncode / LoadImagePNG hand-off (EncoderContext.h:230, EC.cpp:1235):
 * copies Plane::GetPixels() of nPlanes (3 = RGB, 4 = RGBA) planes host -> device into `slot` and resets
 * the slot's analysis state (the reference allocates its state planes lazily per image, EC.cpp:3739-3749). */
int  yk_set_image(yk_ctx* ctx, int slot, const int32_t* const* planes, int nPlanes, int w, int h);
/* How yk_set_image moves the samples: packedU8 != 0 (default) packs the int32 Plane samples to bytes on the host
 * (threads) and uploads a quarter of the bytes; 0 uploads the int32 planes as they are.  Results are identical.  An
 * image with a sample outside 0..255 (signed chroma planes) goes up as int32 in either mode: yk_range_dyn takes it, the
 * alpha / gradient / 1-D range stages return YK_ERR_RANGE for it. */
int  yk_set_upload_format(yk_ctx* ctx, int packedU8);
/* Same, planes already resident in device memory (borrowed, not copied; row pitch == w). */
int  yk_set_image_device(yk_ctx* ctx, int slot, const int32_t* const* devPlanes, int nPlanes, int w, int h);
/* The way in for a decoded image as PNG / JPEG decoders (and Image::LoadPNG before it fills the planes, Image.cpp:200-229)
 * hold it: interleaved 8-bit samples, `channels` bytes per pixel (3 = R,G,B; 4 = R,G,B,A), rows `rowBytes` apart (>= w *
 * channels, any value).  nPlanes = 3 or `channels` (4 channels with nPlanes 3: alpha ignored).  The bytes move as they are
 * (4 or 3 per pixel, no host work) and yk_k_unpack8 splits them into the slot's own packed planes on the device; no byte
 * past the last pixel, rowBytes * (h - 1) + w * channels, is read.
 * Host variant: pinned memory (yk_host_alloc) is read by DMA asynchronously and must not change until the next
 * synchronising call on the context; pageable memory works at the driver's staged rate.
 * Device variant: read by a kernel on the context's stream; the caller orders its own writes before it (yk_set_stream
 * or a sync).  Not borrowed: the buffer may be reused once that kernel has run.
 * Both leave the slot exactly as a packed yk_set_image of the same samples does (so such slots batch with packed uploads).
 * No sample can be out of range.  YK_ERR_ARG: NULL pointer, channels not 3 / 4, nPlanes not 3 / channels, rowBytes
 * < w * channels, or w / h as for yk_set_image; YK_ERR_CAPACITY as for yk_set_image. */
int  yk_set_image_interleaved(yk_ctx* ctx, int slot, const uint8_t* pixels, size_t rowBytes, int channels, int nPlanes, int w, int h);
int  yk_set_image_interleaved_device(yk_ctx* ctx, int slot, const uint8_t* devPixels, size_t rowBytes, int channels, int nPlanes, int w, int h);
/* Device pointer of plane `p` of `slot` (so a caller can fill it in place); NULL on error. */
int32_t* yk_device_plane(yk_ctx* ctx, int slot, int p);
int  yk_reset_state(yk_ctx* ctx, int slot);
int  yk_reset_states(yk_ctx* ctx, int slot0, int nSlots);     /* the same for a batch of slots, one clear */

/* ---- the fused hot path -------------------------------------------------------------------------------
 * Runs, for slots [slot0, slot0+nSlots) (all the same size), on the device, leaving results in HBM:
 *   YK_STAGE_ALPHA     MipPrefilter(true)                          EC.cpp:1257-1427 (quadRecursion 357-430)
 *   YK_STAGE_GRADIENT  the 7 FittingQuadSmooth passes in Convert()'s order   EC.cpp:3710-4235, 9057-9093
 *   YK_STAGE_RANGE1D   DynamicTileCompressor for R, G, B            EC.cpp:8398-8522
 *   YK_STAGE_RANGEDYN  DynamicTileEncode (full-resolution planes)   EC.cpp:4365-4503
 * The per-stage getters below copy the named results to host buffers. */
#define YK_STAGE_ALPHA     1
#define YK_STAGE_GRADIENT  2
#define YK_STAGE_RANGE1D   4
#define YK_STAGE_RANGEDYN  8
#define YK_STAGE_RANGEDYN3 16   /* DynamicTileEncode(mode3BitOnly = true) instead of the 6-mode search */
int  yk_analyze(yk_ctx* ctx, int slot0, int nSlots, int stages, int rejectFactor);

/* ---- stage-by-stage entry points (what the patched member bodies call) ------------------------------- */

/* void EncoderContext::MipPrefilter(bool active)  — EncoderContext.h:332, EC.cpp:1257.
 * bitmap: ceil(tw*th/8) bytes of the kept-tile bbox, bit i (row-major, LSB first) = tile kept (EC.cpp:1317-1327);
 * boundPx = boundX0,boundY0,boundX1,boundY1; wroteChunk = 1 when the reference would write the 'MIPM'
 * chunk (bbox != full image, EC.cpp:1294), chunkBBoxTiles = MipmapHeader.bbox {x,y,w,h} in 16-px tiles.
 * Outside the reference's own domain (w == h == 2^k >= 16) the same per-16x16 rule is applied.
 * Runs the stage if yk_analyze has not already. */
int  yk_alpha_reject(yk_ctx* ctx, int slot, uint8_t* bitmap, int bitmapCap, int* bitmapBytes, int boundPx[4],
                     int* remainingPixels, int* wroteChunk, int chunkBBoxTiles[4]);

/* void EncoderContext::PrepareQuadSmooth()  — EncoderContext.h:327, EC.cpp:2796 (an empty stub in the
 * reference; its state is created lazily in FittingQuadSmooth).  Here: runs all 7 passes in one fused
 * launch sequence so the FittingQuadSmooth calls that follow only fetch their results. */
int  yk_prepare_quad_smooth(yk_ctx* ctx, int slot, int rejectFactor);

/* int EncoderContext::FittingQuadSmooth(rejectFactor, R, G, B, testOutput, false, shX, shY)
 *   — EncoderContext.h:329, EC.cpp:3710; the part before the host tail (EC.cpp:3810-4235).
 * bitmap  = pFillBitMap (getBitmapSwizzleSize()/8 bytes, swizzled bit order, EC.cpp:3770-3777, 4026)
 * rgb     = rgbStream handed to PaletteCompressor (EC.cpp:4115-4132, 4279), *rgbBytes its length
 * bbox    = minX,minY,maxX,maxY of accepted tiles (EC.cpp:4039-4042; {w,h,0,0} when none)
 * tileDone = the function's return value.
 * If the pass was already produced by yk_prepare_quad_smooth/yk_analyze with the same rejectFactor and it
 * is the next pass in Convert()'s order, results are fetched; otherwise the single pass is run on the
 * current state (any order of calls is legal, as in the reference). */
int  yk_gradient_pass(yk_ctx* ctx, int slot, int rejectFactor, int shX, int shY,
                      uint8_t* bitmap, int bitmapCap, int* bitmapBytes,
                      uint8_t* rgb, int rgbCap, int* rgbBytes, int bbox[4], int* tileDone);

/* u8* EncoderContext::DynamicTileCompressor(stream, src = plane, map = mapSmoothTile[plane], debug)
 *   — EncoderContext.h:236, EC.cpp:8398; globals streamType/pType (EC.cpp:8217-8218) become `type`.
 * idx: index bytes 0..16 appended for this plane; type: {color0, minCol, delta} per coded tile. */
int  yk_range1d(yk_ctx* ctx, int slot, int plane, uint8_t* idx, int idxCap, int* idxBytes,
                uint8_t* type, int typeCap, int* typeBytes);

/* int EncoderContext::DynamicTileEncode(mode3BitOnly, plane, dst, false, false, false, false)
 *   — EncoderContext.h:370, EC.cpp:4365; the part before the ZSTD tail (EC.cpp:4365-4503).
 * nibbles: packed 4-bit codes, low nibble first, continuous across tiles (EC.cpp:1174-1190), *nNibbles codes;
 * defs: EncodeTileType(type, range7, base6) u16 per tile with >= 1 valid pixel (include/YAIK_private.h:358);
 * constraint: PlaneTile.bbox {x,y,w,h} (EC.cpp:4386-4391); dst (optional, w*h int32): written only at
 * valid pixels with the decoded value, as the reference does (EC.cpp:4448-4457). */
int  yk_range_dyn(yk_ctx* ctx, int slot, int plane, int mode3BitOnly, uint8_t* nibbles, int nibCap, int* nNibbles,
                  uint16_t* defs, int defsCap, int* nDefs, int constraint[4], int32_t* dst);

/* Chroma front-end of the range stage (SURVEY.md 8f row 3; the pipeline Convert() holds at EC.cpp:9539-9545):
 *
 * yk_chroma_prepare = EncoderContext::convRGB2YCoCg(true) + chromaReduction() (EC.cpp:2766-2782), i.e.
 *   Image::ConvertToRGB2YCoCg (Image.cpp:285-321, RGBtoYCoCg EC.cpp:53-67) and Plane::SampleDown (Plane.cpp:278-369)
 *   of Co and of Cg, in one kernel over the slot's colour planes.  half = {halfCoW, halfCoH, halfCgW, halfCgH}
 *   (EncoderContext.h:265-271; the CLI sets {1,0,1,0}, ImageEncoder.cpp:175-181); downMode = EDownSample of Co, Cg
 *   (framework.h:60-66: 0 NEAREST_TL, 1 NEAREST_BR, 2 AVERAGE_BOX, 3 MAX_BOX, 4 MIN_BOX).  NEAREST_BR / MAX_BOX /
 *   MIN_BOX with ONE axis halved read past the plane in the reference: YK_ERR_UNSUPPORTED.  The planes stay on the device.
 * yk_chroma_plane: which = 0 Y (YCoCgImg plane 0), 1 workCo, 2 workCg; out may be NULL to ask for the size only.
 * yk_range_dyn_chroma = DynamicTileEncode(mode3BitOnly, Y | workCo | workCg, dst, isCo, isCg, isHalfX, isHalfY)
 *   (EC.cpp:4365-4503) with the flags that belong to `which`: the constraint box is halved on the reduced axes
 *   (EC.cpp:4393-4401), both validity rules of the reduced planes are the reference's (min/max: Plane.cpp:528-555 with
 *   its row stride, coding: EC.cpp:831-861), chroma blocks with a negative minimum are written to dst minus 128 and
 *   reduced planes land on dst (full size, w*h int32) at their top-left full-size position only (EC.cpp:4441-4502).
 *   Convert() calls it with mode3BitOnly = 0, 0, 1 for Y, Co, Cg.  Needs w, h (and the reduced sizes) to be multiples of 8. */
int  yk_chroma_prepare(yk_ctx* ctx, int slot, const int half[4], const int downMode[2]);
int  yk_chroma_plane(yk_ctx* ctx, int slot, int which, int32_t* out, int* outW, int* outH);
int  yk_range_dyn_chroma(yk_ctx* ctx, int slot, int which, int mode3BitOnly, uint8_t* nibbles, int nibCap, int* nNibbles,
                         uint16_t* defs, int defsCap, int* nDefs, int constraint[4], int32_t* dst);

/* Expands the compact device state into the reference's int32 state planes so later reference stages
 * (3D LUT search, debug PNGs) keep working: smoothMap, mapSmoothTile[3] (w*h each), mappedRGB[3]
 * ((w+1)*(h+1) each), mipmapMask, recon = testOutput planes (w*h each) — EncoderContext.h:300-323.
 * Any pointer may be NULL. */
int  yk_download_state(yk_ctx* ctx, int slot, int32_t* smoothMap, int32_t* const* mapSmoothTile,
                       int32_t* const* mappedRGB, int32_t* mipmapMask, int32_t* const* recon);

/* Every result of the last run on `slot` with two synchronisations and no per-stream call: the pointers lead into a
 * pinned host arena owned by the context and stay valid until the next run / image on that slot.  Passes that were not
 * part of the run have NULL pointers; the alpha block is filled when the alpha stage ran (alphaValid).  Same contents
 * as the per-stage getters above. */
typedef struct yk_results {
    const uint8_t* bitmap[YK_NUM_PASSES]; int bitmapBytes[YK_NUM_PASSES];
    const uint8_t* rgb[YK_NUM_PASSES];    int rgbBytes[YK_NUM_PASSES];
    int tileDone[YK_NUM_PASSES]; int bbox[YK_NUM_PASSES][4];
    const uint8_t* r2Idx[3]; const uint8_t* r2Type[3]; int r2IdxBytes, r2TypeBytes;      /* per plane */
    int alphaValid; const uint8_t* alphaBitmap; int alphaBitmapBytes; int alphaBound[4]; int alphaRemaining, alphaWroteChunk; int alphaChunkBBox[4];
} yk_results;
int  yk_fetch_all(yk_ctx* ctx, int slot, yk_results* out);

/* Bytes of result streams the last yk_analyze left in HBM for `slot` (for the roofline's algorithmic
 * byte count): [0] bitmaps, [1] rgb streams, [2] R2 idx, [3] R2 type, [4] alpha tile bitmap, [5] R1. */
int  yk_result_bytes(yk_ctx* ctx, int slot, long long out[6]);
/* Number of kernel launches enqueued by this context since creation. */
long long yk_launch_count(yk_ctx* ctx);

/* Per-kernel device time: while enabled, every launch is bracketed by a CUDA event pair on the launching stream;
 * yk_profile_read synchronises, sums the elapsed milliseconds per kernel (0 yk_k_analyze, 1 yk_k_emit, 2 yk_k_owner,
 * 3 yk_k_r1_encode, 4 yk_k_chroma, 5 yk_k_unpack8; the other entries are unused) with their launch counts, and clears the record.  Used by bench.py's roofline figure. */
int  yk_profile(yk_ctx* ctx, int enable);
int  yk_profile_read(yk_ctx* ctx, double ms[8], long long count[8]);

/* ---- multi-GPU: tile-row strips of one large image (SURVEY.md §8e; BASELINE.json configs[3]) -------------
 * The reference has no counterpart (Convert() walks one image on one thread); this is the partition of
 * FittingQuadSmooth / DynamicTileCompressor over GPUs.  A strip holds rows [y0, y0+h) of an image of height
 * imgH (y0 a multiple of 64 = the largest swizzle block, h a multiple of 64 except for the last strip), as
 * an ordinary image of its own context (yk_set_image), then:
 *   yk_strip_config      declares the strip's place and allocates its halo-in buffer
 *   (exchange 1)         every strip copies its first pixel row (3 planes) into the halo of the strip above:
 *                        the clamped bottom corners of that strip's last tile row become the real samples
 *   yk_strip_phase 0     accept decisions + range stage of the strip (yk_k_analyze)
 *   (exchange 2)         every strip copies the touch words of its top / bottom boundary lattice row into
 *                        the halo of the strip above / below, so both sides agree on who emits those corners
 *                        (a tile of the upper strip precedes every tile of the lower strip in a pass's stream)
 *   yk_strip_phase 1     corner ownership + rgbStream emission + range-stream gather
 * and the per-pass getters return the strip's part: bitmaps are consecutive byte ranges of the image's
 * bitmaps, rgb / range streams concatenate in strip order, TileDone adds up, boxes merge (they are in image
 * coordinates).  The two exchanges are plain device-to-device copies (NVLink P2P through CUDA IPC between
 * the per-GPU processes), never a collective.  Only the fused 7-pass form on a fresh state is provided, plus
 * DynamicTileEncode of R, G, B (yk_strip_range_dyn below); the chroma front-end is not provided for strips. */
typedef struct yk_strip_halo {
    void*  haloIn;                 /* one device allocation of this strip, written by its neighbours */
    size_t haloBytes;
    size_t pixelRowInOffset, pixelRowBytes;      /* 3 planes x w samples (int32, or bytes after a packed upload): first pixel row of the strip below */
    size_t pixelRowStride;                       /* plane p of that row starts at pixelRowInOffset + p * pixelRowStride */
    size_t touchInTopOffset, touchInBottomOffset, touchBytes;   /* latW u32 each: boundary touch words of the strip above / below */
    const void* pixelRowOut[3];    /* this strip's first pixel row, per colour plane (planeRowBytes each) */
    size_t planeRowBytes;
    const void* touchOutTop;       /* this strip's touch words of its top / bottom boundary lattice row */
    const void* touchOutBottom;
} yk_strip_halo;
int  yk_strip_config(yk_ctx* ctx, int slot, int imgH, int y0);
int  yk_strip_halo_ptrs(yk_ctx* ctx, int slot, yk_strip_halo* out);
int  yk_strip_phase(yk_ctx* ctx, int slot, int phase, int rejectFactor);  /* 0 = accept phase, 1 = emission phase */
/* DynamicTileEncode (EC.cpp:4365-4503) of the strip's rows, R, G and B in one launch pair, after phase 0 (an 8x8 block
 * needs only its own samples, its cells' claimed bits and the alpha mask, so it needs no halo).  The strip codes exactly
 * the blocks of the whole image's LeftRightOrder walk whose top row it holds, with the image's geometry (constraint box,
 * block sizes).  imageBoundPx: the strip set's merged alpha box for 4 planes (strips.merge_alpha / yk_alpha_assemble),
 * NULL for 3 planes (the whole image); the alpha mask applies unless that box is the whole image (EC.cpp:1400-1403).
 * Enqueued only, no synchronisation.  yk_range_dyn(..., dst = NULL) on the strip then returns the strip's part of each
 * plane's streams: nibbles and defs start at 0 for every strip, and the strips' parts concatenated in strip order are the
 * image's streams (every part has an even nibble count); `constraint` is the image's box.  yk_range_dyn on a strip returns
 * YK_ERR_STATE if the strip was not coded in that mode and YK_ERR_UNSUPPORTED for dst != NULL.
 * YK_ERR_ARG: the box is empty or outside [0, w) x [0, imgH), a box for 3 planes, none for 4, or w / imgH not multiples
 * of 8 or below 32.  YK_ERR_STATE: not a strip, or phase 0 has not run on this image.
 * Not provided for strips: the chroma front-end (the reduced planes' min/max rule reads mask rows of other strips,
 * Plane.cpp:516) and the write-back plane. */
int  yk_strip_range_dyn(yk_ctx* ctx, int slot, int mode3BitOnly, const int imageBoundPx[4]);
/* The same protocol without the host in the loop: after yk_strip_config on every strip (and one host barrier, so that
 * every halo is cleared before a neighbour writes into it) each strip is told where its neighbours' halo allocations
 * are mapped in this process (their haloIn, direct or through yk_ipc_open; NULL where there is no neighbour), and
 * yk_strip_run then enqueues a whole image on the strip's stream: reset, exchange 1, phase 0, exchange 2, phase 1.
 * The exchanges are peer copies followed by a one-thread kernel that publishes an epoch number in the neighbour's halo;
 * a one-thread kernel on the receiving stream waits for it, and a strip does not start the next image before both
 * neighbours have finished the current one.  Images can be enqueued back to back; the planes must stay what
 * yk_set_image / yk_set_image_device made them.  yk_strip_set_peers also makes the R1 tables resident (it synchronises
 * the stream on first use); yk_strip_run never makes the host wait.
 * yk_strip_run_stages: stages = 0, YK_STAGE_RANGEDYN or YK_STAGE_RANGEDYN3 (any other bit: YK_ERR_ARG) adds
 * DynamicTileEncode of the strip (as yk_strip_range_dyn with the whole image as box) between exchange 2 and phase 1,
 * while the touch words travel.  3 planes only: with R1, an RGBA strip returns YK_ERR_UNSUPPORTED before anything is
 * enqueued (its alpha box is a reduction over all strips, not a neighbour exchange).  yk_strip_run = stages 0. */
int  yk_strip_set_peers(yk_ctx* ctx, int slot, void* aboveHalo, void* belowHalo);
int  yk_strip_run(yk_ctx* ctx, int slot, int rejectFactor);
int  yk_strip_run_stages(yk_ctx* ctx, int slot, int rejectFactor, int stages);
/* All strips of an image driven by one process (ctxs[k] = strip k, top to bottom, on one or several GPUs): link every
 * strip to its neighbours (peer access is enabled between their devices), enqueue one image on every strip. */
int  yk_strips_link(yk_ctx* const* ctxs, int n, int slot);
int  yk_strips_run(yk_ctx* const* ctxs, int n, int slot, int rejectFactor);
int  yk_strips_run_stages(yk_ctx* const* ctxs, int n, int slot, int rejectFactor, int stages);    /* every strip checked before any is enqueued */
/* Alpha stage of a strip set (yk_alpha_reject serves whole images): the per-16x16-tile "has a non-zero alpha sample" bytes of
 * one strip ([tilesH][tilesW], row-major) with the box of its kept tiles in image coordinates, and the assembly of
 * MipPrefilter's results (EC.cpp:1287-1403) from the strips' arrays one after the other and the merged box: host code. */
int  yk_alpha_kept(yk_ctx* ctx, int slot, uint8_t* kept, int keptCap, int* tilesW, int* tilesH, int boundPx[4], int* keptTiles);
int  yk_alpha_assemble(const uint8_t* kept, int tilesW, int tilesH, int w, int h, const int boundPx[4],
                       uint8_t* bitmap, int bitmapCap, int* bitmapBytes, int* remainingPixels, int* wroteChunk, int chunkBBoxTiles[4]);

/* Plumbing for the exchanges: CUDA IPC handle of a device allocation (64 bytes, to be sent to the neighbour's
 * process by any host channel), mapping it in this process, and an asynchronous device-to-device copy on the
 * context's stream (peer access is enabled lazily by the mapping).  yk_copy_to_host / yk_copy_from_host are the
 * host-staged alternative when the GPUs have no peer access. */
int  yk_ipc_export(const void* devPtr, unsigned char handle[64]);
int  yk_ipc_open(yk_ctx* ctx, const unsigned char handle[64], void** devPtr);
int  yk_ipc_close(yk_ctx* ctx, void* devPtr);
int  yk_copy_async(yk_ctx* ctx, void* dst, const void* src, size_t bytes);
int  yk_copy_to_host(yk_ctx* ctx, void* hostDst, const void* devSrc, size_t bytes);
int  yk_copy_from_host(yk_ctx* ctx, void* devDst, const void* hostSrc, size_t bytes);

/* ---- host tails behind the analysis stage (SURVEY.md 8f rows 1-2): plain host code, no device involved ------
 *
 * PaletteCompressor (EC.cpp:3209-3502), the delta code-book coder of a gradient pass's rgbStream, as an object
 * instead of the reference's globals CodeRGB[100000] / CodeCount (EC.cpp:3216-3217).  The reference never clears that
 * table and FindCodeBook always scans 64 entries (EC.cpp:3248-3255), so its bytes depend on the calls made before
 * (SURVEY.md S10).  YK_PALETTE_BUG_COMPATIBLE reproduces them call for call, starting from a fresh object = a fresh
 * process; YK_PALETTE_DECODABLE only emits indices of the code book it writes (what PaletteDecompressor can read).
 * yk_palette_compress returns YK_ERR_CAPACITY where the reference's WriteRAW would overflow `maxSize`. */
#define YK_PALETTE_BUG_COMPATIBLE 0
#define YK_PALETTE_DECODABLE      1
typedef struct yk_palette yk_palette;
yk_palette* yk_palette_create(int mode);
void yk_palette_destroy(yk_palette* p);
void yk_palette_reset(yk_palette* p);
int  yk_palette_compress(yk_palette* p, const uint8_t* rgbStream, int size, uint8_t* out, int outCap, int* outBytes);

/* Chunk serialisers of Convert() with the entropy coder as a callback: compress(user, dst, dstCap, src, srcBytes,
 * level) returns the compressed size, 0 on failure (ZSTD_compress with its arguments in that order; the reference
 * uses level 18, 21 for PLNT).  Every function writes one chunk at dst and returns its size in *n (0 = the reference
 * writes no chunk for these arguments).  Layouts: include/YAIK_private.h:96-118, 172-197, 290-300, 347-356.
 *   yk_chunk_file_header  FileHeader 'YAIK'                                  EC.cpp:9007-9016
 *   yk_chunk_mipm         MipPrefilter's chunk                               EC.cpp:1367-1396
 *   yk_chunk_gtil         FittingQuadSmooth's chunk (runs PaletteCompressor) EC.cpp:4239-4350; bbox = {minX,minY,maxX,maxY}
 *   yk_chunk_1dtl         GenerateDynamicTileChunk                           EC.cpp:8524-8576
 *   yk_chunk_plnt         DynamicTileEncode's chunk                          EC.cpp:4515-4589; planeType 0 Y, 1 Co, 2 Cg
 *   yk_chunk_end          0xDEADBEEF                                         EC.cpp:9779-9782 */
typedef size_t (*yk_compress_fn)(void* user, void* dst, size_t dstCap, const void* src, size_t srcBytes, int level);
int  yk_chunk_file_header(uint8_t* dst, size_t cap, size_t* n, int width, int height, int hasAlpha);
int  yk_chunk_mipm(uint8_t* dst, size_t cap, size_t* n, const int bboxTiles[4], const uint8_t* bitmap, int bitmapBytes);
int  yk_chunk_gtil(uint8_t* dst, size_t cap, size_t* n, yk_palette* palette, yk_compress_fn compress, void* user,
                   int shX, int shY, int planeBits, const int bbox[4], const uint8_t* bitmap, int bitmapBytes,
                   const uint8_t* rgbStream, int rgbBytes, int colorCompression);
int  yk_chunk_1dtl(uint8_t* dst, size_t cap, size_t* n, yk_compress_fn compress, void* user, const uint8_t* idx, int idxBytes,
                   const uint8_t* type, int typeBytes, int compressionColor, int compressionRange);
int  yk_chunk_plnt(uint8_t* dst, size_t cap, size_t* n, yk_compress_fn compress, void* user, const int constraint[4],
                   const uint16_t* defs, int nDefs, const uint8_t* nibbles, int nNibbles, int planeType, int halfX, int halfY);
int  yk_chunk_end(uint8_t* dst, size_t cap, size_t* n);

#ifdef __cplusplus
}
#endif
#endif
