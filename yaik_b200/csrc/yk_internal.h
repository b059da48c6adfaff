// Internal declarations shared by the kernels (yk_kernels.cu) and the C-ABI layer (yk_api.cu).
// Vocabulary follows the reference (KLab/YAIK): planes, tiles, swizzle blocks, passes, streams.
#pragma once
#include <stdint.h>
#include <stddef.h>
#include <limits.h>

#ifndef YK_EMULATE
#include <cuda_runtime.h>
#define YK_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#endif

#define YK_NPASS 7
#define YK_REGION 64            // the largest swizzle block (YAIK_private.h:212-276): regions tile the image, strips start on them
#define YK_THREADS 256          // CTA size of the auxiliary kernels (state download, DynamicTileEncode)

// Swizzle geometry of pass id p (HeaderGradientTile::getSwizzleSize, include/YAIK_private.h:212-276),
// in Convert()'s order (EC.cpp:9057-9093): 16x16 16x8 8x16 8x8 8x4 4x8 4x4.
struct YkPassGeom { int shx, shy, bw, bh, bits; };
#define YK_PASS_TABLE { {4,4,64,64,16}, {4,3,64,64,32}, {3,4,64,64,32}, {3,3,64,64,64}, {3,2,64,32,64}, {2,3,32,64,64}, {2,2,32,32,64} }

// per-pass counters written by the analysis kernels (ints)
enum { YK_ST_TILEDONE = 0, YK_ST_MINX, YK_ST_MINY, YK_ST_MAXX, YK_ST_MAXY, YK_ST_RGBBYTES, YK_ST_PAD0, YK_ST_PAD1, YK_ST_STRIDE };
// per-slot header ints (device memory, zeroed/initialised before each run)
enum {
    YK_HD_ERR = 0,                 // bit0: sample outside 0..255
    YK_HD_ALPHA_KEPT0,             // alpha stage: kept tiles, then their box (count first, like a pass's counters)
    YK_HD_ALPHA_MINX, YK_HD_ALPHA_MINY, YK_HD_ALPHA_MAXX, YK_HD_ALPHA_MAXY,
    YK_HD_R2_CHUNKS, YK_HD_R2_TILES,        // totals from the scan: 16-byte chunks per plane, coded tiles per plane
    YK_HD_R1_NIB0, YK_HD_R1_NIB1, YK_HD_R1_NIB2, YK_HD_R1_DEF0, YK_HD_R1_DEF1, YK_HD_R1_DEF2,
    YK_HD_TICKET_ANALYZE,          // work ticket: regions of the persistent analysis kernel
    YK_HD_PASS0 = 16,              // YK_NPASS * YK_ST_STRIDE ints
    YK_HD_INTS = YK_HD_PASS0 + YK_NPASS * YK_ST_STRIDE
};

// TMA descriptor of one int32 plane as a 2-D tensor [h][w] (a CUtensorMap: 128 bytes, 64-byte aligned), encoded on
// the host by cuTensorMapEncodeTiled.  Box = 132 x 17 samples for the colour planes (one macro-tile row of two
// neighbouring 64x64 regions plus its right / bottom corner samples: the TMA unit's cost is per box row, so rows are
// made long), 128 x 16 for alpha; out-of-image samples arrive as zeros and are never used unclamped.
struct alignas(64) YkTmap { unsigned long long opaque[16]; };
#ifndef YK_EMIT_THREADS
#define YK_EMIT_THREADS 512    // threads of a yk_k_emit CTA == nibble words / range tiles per group (host and device agree on it)
#endif
#ifndef YK_SUPER
#define YK_SUPER 32             // groups per super-group: the second level of the group totals
#endif
#define YK_UNIT_W 128           // pixels a unit of the analysis kernel is wide (two regions)
#define YK_RAW_PITCH 132        // samples per row of a staged colour box
#define YK_RAW_ROWS 17

// Device-visible description of one slot (one image + all results of its analysis).
#define YK_U8_BOX 144           // bytes per row of a staged colour box of a packed (u8) plane: 128 + corner column, 16-byte granular

struct alignas(128) YkSlotDev {
    YkTmap tmap[4];             // per plane (R, G, B, alpha): int32 planes, or the packed u8 planes when isU8
    const int32_t* plane[4];    // int32 row-major planes, pitch == w (Plane::GetPixels(), framework.h:81); with isU8 they are
                                //   only filled on demand (yk_k_expand) for the kernels outside the hot path
    const uint8_t* planeU8[4];  // packed upload (yk_set_image): one byte per sample, row pitch pitchU8
    int isU8, pitchU8;
    const void* rowBelow[3];    // strip mode: the pixel row under the strip (w samples, int32 or u8 like the planes), else NULL
    int w, h, nPlanes;
    int nbx, nby;               // 64x64 regions
    int imgH, y0;               // strip mode: height of the whole image / first row of this strip (else h, 0)
    int hasAbove, hasBelow;     // strip mode: there is a strip above / below this one
    const uint32_t* touchInTop;     // strip mode: touch words of the boundary lattice row as the strip above / below saw them
    const uint32_t* touchInBottom;  //   (latW words each, written by the neighbour over NVLink P2P between the two phases)
    int latW, latH;             // lattice of 4-pixel points: w/4+1, h/4+1
    // ---- compact state (replaces the reference's int32 state planes, EncoderContext.h:300-323)
    uint16_t* cellMask;         // [h/4][nbx]   bit i = 4x4 cell (16*bx+i) claimed   == smoothMap / mapSmoothTile != 0
    uint32_t* touchMap;         // [latH][latW] per lattice point: bit 4*rp+k = in pass position rp of the running launch an
                                //   accepted tile has this point as corner k (0 TL,1 TR,2 BL,3 BR); bit 31 = claimed by an
                                //   earlier launch.  != 0  ==  mappedRGB != 0
    uint8_t*  alphaKept;        // [ceil(h/16)][ceil(w/16)] 1 = tile has a non-zero alpha sample
    int*      hdr;              // YK_HD_INTS ints
    // ---- gradient results
    uint8_t*  bitmap[YK_NPASS];     // pFillBitMap in the reference's swizzled layout
    uint32_t* rgbTot[YK_NPASS];     // per group of YK_EMIT_THREADS nibble words: rgb bytes its tiles emit (added by yk_k_owner)
    uint32_t* rgbSup[YK_NPASS];     //   the same per super-group of YK_SUPER groups
    uint8_t*  rgb[YK_NPASS];        // rgbStream
    uint8_t*  latRGB;               // [latH][latW][3]  CompressF(Round6(clamped pixel),250) at every lattice point
    uint32_t* emitNib[YK_NPASS];    // per tile in stream order 4 bits: which of TL,TR,BL,BR the tile emits (8 tiles per word)
    // ---- range stage R2 (DynamicTileCompressor)
    unsigned long long* r2Tot;      // per group of YK_EMIT_THREADS tiles (row-major tile order): chunks << 32 | coded tiles (added by yk_k_owner)
    unsigned long long* r2Sup;      //   the same per super-group of YK_SUPER groups
    uint8_t*  r2Raw[3];         // [h/8][w/8][64] index bytes of every coded tile at a fixed place (written by the analysis kernel)
    uint32_t* r2RawType[3];     // [h/8][w/8] color0 | minCol << 8 | delta << 16
    uint8_t*  r2Idx[3];         // the streams in the reference's order (gathered by yk_k_emit)
    uint8_t*  r2Type[3];
    // ---- range stage R1 (DynamicTileEncode)
    unsigned long long* r1Status;   // look-back words of yk_k_r1_offsets' units (256 blocks of the walk each) + the unit ticket; zeroed per call
    void*     r1List;           // the blocks that hold valid pixels, in walk order (16 bytes each, see yk_k_r1_offsets)
    uint32_t* r1Nib[3];         // nibble stream (two nibbles per byte, written pairwise)
    uint16_t* r1Defs[3];
    int       alphaReset;       // set by the host after the alpha stage: bbox == full image -> mask all 255 (EC.cpp:1400-1403)
    int       alphaValid;       // alpha stage has been run for this image
};

struct YkRun {
    int nPasses;
    int passId[YK_NPASS];       // which passes this launch runs, in order
    int rejectFactor;
    int doAlpha;
    int doR2;                   // code the DynamicTileCompressor tiles of every region after its cascade
    int endgameUnits;           // units per CTA at the end of a launch that are taken on demand instead of ahead (load balance of the tail)
    int fresh;                  // no cell is claimed yet (first gradient launch after yk_reset_state): cellMask need not be read
};

// The box (L, T, R, B) of the tiles the alpha stage kept, from the image header (MipPrefilter, EC.cpp:1287-1291); false and
// an empty box when it kept none.  The analysis keeps w - L and INT_MAX / 2 - T so that every update is an atomicMax.
static __host__ __device__ inline bool yk_alpha_box(const int* hdr, int w, int box[4]) {
    const bool any = hdr[YK_HD_ALPHA_KEPT0] > 0;
    box[0] = any ? w - hdr[YK_HD_ALPHA_MINX] : 0; box[1] = any ? INT_MAX / 2 - hdr[YK_HD_ALPHA_MINY] : 0;
    box[2] = any ? hdr[YK_HD_ALPHA_MAXX] : 0; box[3] = any ? hdr[YK_HD_ALPHA_MAXY] : 0;
    return any;
}
// a box over the whole image discards the alpha stage's rejection: mipmapMask stays 255 everywhere (EC.cpp:1294, 1400-1403)
static __host__ __device__ inline bool yk_box_is_image(const int box[4], int w, int h) {
    return box[0] == 0 && box[1] == 0 && box[2] == w && box[3] == h;
}

// Range stage R1 (DynamicTileEncode) tables, built by the host (DynamicTile::buildTable, EC.cpp:625-699), see yk_kernels.cu
#define YK_R1_BASE_MAX 224          // the block minimum is clamped to 0..224 and quantised to base6 = 0..63
#define YK_R1_R7_ROW 224            // range7 per base6 for the clamped differences 32..255
#define YK_R1_R7MAX 176             // range7 values the LUTs cover (above 127 for bases close to 224: a reference quirk)
#define YK_R1_LUT_INTS 144          // six LUTs (16,16,16,8,8,8 entries) and their decision thresholds
#define YK_R1_RTAB_VALUES 384       // sample values of the per-value table: -128..255, shifted by 128 when the minimum is negative
#define YK_R1_RTAB_R7 128           // range7 values the per-value table covers: every entry of those LUTs is a byte

// The walk of LeftRightOrder (framework.h:228-256) over the 8-aligned bound box (EC.cpp:4386-4401), halved on the
// reduced axes of a plane of ph rows: rows of nbw = ceil(cw / 8) blocks while y < cy + ch, then one more block at the
// start of the next row when that row still lies inside the plane (HasNextBlock tests `y < h` after the wrap).
// A launch codes blocks b0 .. b0 + nBlocks - 1 of the walk (all of them, or the window of a tile-row strip).
struct YkR1Walk { int cx, cy, cw, ch, nbw, nBlocks, b0; };
static __host__ __device__ inline YkR1Walk yk_r1_walk(const int box[4], int ph, int shX, int shY) {
    YkR1Walk g;
    g.cx = (box[0] >> 3) << 3; g.cy = (box[1] >> 3) << 3;                              // EC.cpp:4386-4391
    g.cw = (((box[2] + 7) >> 3) << 3) - g.cx; g.ch = (((box[3] + 7) >> 3) << 3) - g.cy;
    g.cx >>= shX; g.cw >>= shX; g.cy >>= shY; g.ch >>= shY;                            // EC.cpp:4393-4401
    g.nbw = (g.cw + 7) >> 3;
    const int rows = (g.ch + 7) >> 3;
    g.nBlocks = g.nbw * rows;
    if (g.nBlocks > 0 && g.cy + 8 * rows < ph) g.nBlocks += 1;
    g.b0 = 0;
    return g;
}
// The window of a whole-image walk g that a tile-row strip of rows [y0, y0 + h) codes: the blocks whose top row (image
// coordinates) lies in the strip, the extra block after the last row included.  Rows are whole walk rows, so the
// strips' windows cut the walk into consecutive pieces.
static __host__ __device__ inline YkR1Walk yk_r1_window(YkR1Walk g, int y0, int h) {
    const int total = g.nBlocks;
    const int r0 = y0 <= g.cy ? 0 : (y0 - g.cy + 7) >> 3, r1 = y0 + h <= g.cy ? 0 : (y0 + h - g.cy + 7) >> 3;     // first walk row at or below y0, y0 + h
    const long long first = (long long)r0 * g.nbw, end = (long long)r1 * g.nbw;
    g.b0 = (int)(first < total ? first : total);
    g.nBlocks = (int)(end < total ? end : total) - g.b0;
    return g;
}

#ifdef __cplusplus
extern "C++" {
#endif
// launch wrappers (yk_kernels.cu); `slots` is a device array, grid.y indexes it from slot0
int  yk_analyze_setup(int* numSMs);
int  yk_preload_analyze();              // force-load every kernel of a translation unit (see yk_analyze.cu); return a cudaError_t
int  yk_preload_emit();
int  yk_preload_aux();      // opt-in shared memory of the persistent kernel; returns a cudaError_t
void yk_launch_analyze(const YkSlotDev* slotsDev, int slot0, int nSlots, int nRegions, int gridCtas, bool packedU8, const YkRun& run, cudaStream_t st);   // nRegions: of one image (nbx * nby)
void yk_launch_expand(const YkSlotDev* slotsDev, int slot, int nPlanes, int w, int h, int32_t* const* dst, cudaStream_t st);
// interleaved 8-bit pixels (channels 3 or 4, rows rowBytes apart) -> nPlanes packed planes of row pitch `pitch` (yk_k_unpack8)
struct YkUnpackArgs { const uint8_t* src; size_t rowBytes; int nPlanes, w, h, pitch; uint8_t* dst[4]; };
void yk_launch_unpack8(const YkUnpackArgs& a, int channels, cudaStream_t st);
void yk_launch_fold_touch(const YkSlotDev* slotsDev, int slot0, int nSlots, int nWords, cudaStream_t st);
// one-thread kernels on a strip's stream: publish / wait for an epoch number in (peer-mapped) halo memory
void yk_launch_flag_set(unsigned* a, unsigned* b, unsigned value, cudaStream_t st);
void yk_launch_flag_wait(const unsigned* a, const unsigned* b, unsigned value, cudaStream_t st);
void yk_launch_owner(const YkSlotDev* slotsDev, int slot0, int nSlots, int nPoints, bool owners, const YkRun& run, cudaStream_t st);   // owners: resolve corner ownership; run.doR2: count the range tiles
void yk_launch_emit(const YkSlotDev* slotsDev, int slot0, int nSlots, int gradGroups, int r2Groups, const YkRun& run, cudaStream_t st);
void yk_launch_state(const YkSlotDev* slotsDev, int slot, int nRegions, int32_t* smoothMap, int32_t* mipmapMask,
                     int32_t* mappedRGB, int32_t* recon0, int32_t* recon1, int32_t* recon2, cudaStream_t st);
// DynamicTileEncode on one plane: the source samples and where the results go
struct YkR1Args {
    const int32_t* src;                  // plane coded: pw x ph int32 samples on the device
    const uint8_t* srcU8; int pitchU8;   // ... or, when not NULL, one byte per sample (a colour plane uploaded packed)
    int32_t* dst;                        // optional write-back plane (w x h int32, full size), else NULL
    int chroma;                          // isCo | isCg
    int out;                             // index of r1Nib / r1Defs / header counters written
};
struct YkChromaArgs { int32_t *y, *co, *cg; int half[4]; int mode[2]; };
// one launch: 1 plane, or the 3 full-resolution colour planes, with the same geometry and validity; fromHdr: the walk is
// derived on the device from the alpha stage's box in the image header (the fused yk_analyze path, no host round trip),
// `walk` is then the largest possible one and sizes the launch
struct YkR1Launch {
    int nJobs, fromHdr, useAlpha, mode3;     // mode3: mode3BitOnly
    int pw, ph, shX, shY;                    // plane size; shX / shY = 1: SampleDown'ed on that axis (isHalfX / isHalfY)
    YkR1Walk walk;
    YkR1Args job[3];
};
void yk_launch_range_dyn_encode(const YkSlotDev* slotsDev, int slot, const YkR1Launch& launch, int numSMs, const int* lutDev, const uint16_t* rtabDev, const int16_t* r7Dev, cudaStream_t st);
void yk_launch_chroma(const YkSlotDev* slotsDev, int slot, int w, int h, const YkChromaArgs& args, cudaStream_t st);
#ifdef __cplusplus
}
#endif
