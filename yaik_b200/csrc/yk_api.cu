// yaik_b200 — the extern "C" layer declared in include/yaik_b200.h: context/slot management, launch sequencing and
// result download.  Host code is C++; all device work goes through the launch wrappers of yk_kernels.cu.
// There is no CPU path here: every compute entry point needs a CUDA device.
#include "../../include/yaik_b200.h"
#include "yk_internal.h"
#define YK_ENDGAME_UNITS 6      // units per CTA at the end of a full-GPU launch that are taken on demand (yk_analyze.cu, producer)

#include <limits.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <string>
#include <vector>
#ifndef YK_EMULATE
#include <cuda.h>               // CUtensorMap types only; the encoder is fetched with cudaGetDriverEntryPoint (no libcuda link)
#endif

// yk_hostpack.cpp
struct YkHostPacker;
YkHostPacker* yk_hostpack_create(int threads);
void yk_hostpack_destroy(YkHostPacker* p);
int yk_hostpack_threads(const YkHostPacker* p);
unsigned yk_hostpack_plane(YkHostPacker* p, const int32_t* src, uint8_t* dst, int w, int h, size_t pitch);

static thread_local std::string g_lastCuda;

#define CK(call)                                                                            \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            g_lastCuda = std::string(#call) + ": " + cudaGetErrorString(e__);               \
            return YK_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

static const YkPassGeom kGeom[YK_NPASS] = YK_PASS_TABLE;

static int pass_id(int shX, int shY) {
    for (int i = 0; i < YK_NPASS; i++) if (kGeom[i].shx == shX && kGeom[i].shy == shY) return i;
    return -1;
}

struct YkSlotHost {
    YkSlotDev d;
    bool haveImage = false, borrowed = false, dirty = true;
    int32_t* owned[4] = { 0, 0, 0, 0 };
    uint8_t* ownedU8[4] = { 0, 0, 0, 0 };     // packed upload: device planes, pinned staging, "staging is free again" event
    uint8_t* stageHost = nullptr; size_t stageBytes = 0;
    cudaEvent_t stageFree = nullptr; bool stageBusy = false;
    bool int32Valid = true;      // owned[] holds the int32 samples (false after a packed upload until yk_k_expand ran)
    uint8_t* arena = nullptr; size_t arenaBytes = 0;     // pinned host copy of every result stream of the last run
    bool harvested = false;
    size_t arBitmap[YK_NPASS], arRgb[YK_NPASS], arIdx[3], arType[3], arKept = 0;
    int arMask = 0; bool arR2 = false, arHasKept = false;
    // what is valid on the device for the current image
    bool k1Ran = false;          // r2Seg / latRGB are current
    bool alphaRan = false, alphaFetched = false;
    bool prepared = false;       // fused 7-pass cascade results present
    int  preparedReject = 0, nextPass = 0;
    bool r2Valid = false;
    bool zeroAClean = false;     // part A of the zero area is still all zero (nothing launched since the reset)
    bool touchDirty = false;     // the touch map holds claims of an earlier launch (needs folding before the next one)
    bool cellsClean = false;     // no gradient pass has run since the state was reset (nothing claimed, bitmaps all zero)
    bool pendingHarvest = false; // a run's header has not been copied back yet
    int  lastRunPasses = 0;      // bit p: pass p was in the last run; bit 8: alpha
    int  rangeErr = 0;
    int32_t* r1DstDev = nullptr;  // write-back plane of DynamicTileEncode (allocated on first use, one plane at a time)
    int  r1Fused = 0;            // DynamicTileEncode results of the three colour planes present from yk_analyze: 1 = six modes, 2 = 3-bit only
    int32_t* chroma[3] = { nullptr, nullptr, nullptr };   // Y, workCo, workCg of the chroma front-end (allocated on first use)
    int  chromaHalf[4] = { 0, 0, 0, 0 };
    bool chromaReady = false;
    int  hdr[YK_HD_INTS];        // harvested copy: per-pass stats of the run that produced them, alpha box, R2 totals
    long long resultBytes[6] = { 0, 0, 0, 0, 0, 0 };
    // alpha results (host)
    int bound[4] = { 0, 0, 0, 0 }, remaining = 0, wroteChunk = 0, chunkBBox[4] = { 0, 0, 0, 0 };
    std::vector<uint8_t> alphaBitmap;
    std::vector<void*> devAllocs;        // every device allocation of the slot (freed by yk_destroy)
    // strip mode: one allocation [3 * w int32 pixel row][latW touch words from above][latW touch words from below]
    uint8_t* haloIn = nullptr; size_t haloBytes = 0;
    size_t haloFlagsOffset = 0;  // five u32 epoch flags written by the neighbours: see yk_strip_run
    void* peerAbove = nullptr; void* peerBelow = nullptr;     // the neighbours' halo allocations as mapped in this process
    unsigned stripEpoch = 0;
    bool strip = false;          // yk_strip_config placed the current image in a strip set
    int  r1Strip = 0;            // DynamicTileEncode of the strip's rows present (yk_strip_range_dyn): 1 = six modes, 2 = 3-bit only
    int  r1StripConstraint[4] = { 0, 0, 0, 0 };     // ... and the image's constraint box it was coded in
};

struct yk_ctx {
    int device = 0, maxW = 0, maxH = 0, maxPlanes = 0, maxSlots = 0;
    cudaStream_t stream = 0; bool ownStream = false;
    YkSlotDev* slotsDev = nullptr;
    std::vector<YkSlotHost> slots;
    // per slot one contiguous zeroable area: part A (header, look-back status words) is cleared before every launch,
    // part B (claimed cells, touch map = the persistent analysis state) only by yk_reset_state
    uint8_t* zeroArea = nullptr; size_t zeroStride = 0, zeroABytes = 0;
    int* lutDev = nullptr;       // R1 tables: LUTs + thresholds, and the per-value entry table (see yk_k_r1_encode)
    uint16_t* rtabDev = nullptr;
    int16_t* r7Dev = nullptr;    // range7 code per (base6, clamped difference)
    int numSMs = 1;              // SMs of the device
    int analysisCtas = 1;        // grid of the persistent analysis kernel (default: one CTA per SM)
    YkHostPacker* packer = nullptr;
    bool packedUpload = true;    // yk_set_image packs Plane samples to bytes on the host before the copy
    long long launches = 0;
    size_t planeCap = 0;
    // optional per-kernel timing with CUDA events on the launching stream (yk_profile)
    bool profile = false;
    std::vector<cudaEvent_t> evA[6], evB[6];      // 0 analyze, 1 emit, 2 owner, 3 r1_encode, 4 chroma, 5 unpack8
    // device copy of the caller's interleaved rows (yk_set_image_interleaved), same row stride; allocated on first use and
    // grown on demand.  One per context is enough: stream order puts every copy into it after the unpack of the previous one.
    // Its base is 256-byte aligned, so 16-byte aligned rows take yk_k_unpack8's vector path whatever the caller's base.
    uint8_t* stage8 = nullptr; size_t stage8Bytes = 0;
    // set while yk_strip_run_stages enqueues: the steps that would make the host wait for the stream (a pageable
    // descriptor upload, a header copy-back, the first upload of the R1 tables) fail with YK_ERR_STATE instead
    bool noHostWait = false;
};

struct YkTimed {        // records an event pair around one launch when profiling is on
    yk_ctx* c; int k;
    YkTimed(yk_ctx* c_, int k_) : c(c_), k(k_) {
        if (c->profile && c->evA[k].size() < 100000) {
            cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
            c->evA[k].push_back(a); c->evB[k].push_back(b);
            cudaEventRecord(a, c->stream);
        } else k = -1;
    }
    ~YkTimed() { if (k >= 0) cudaEventRecord(c->evB[k].back(), c->stream); }
};

extern "C" int yk_abi_version(void) { return 1; }

extern "C" const char* yk_error_string(int code) {
    switch (code) {
    case YK_OK: return "ok";
    case YK_ERR_CUDA: return "CUDA error";
    case YK_ERR_ARG: return "bad argument";
    case YK_ERR_CAPACITY: return "capacity exceeded";
    case YK_ERR_RANGE: return "sample outside 0..255";
    case YK_ERR_STATE: return "wrong call order / no image";
    case YK_ERR_UNSUPPORTED: return "unsupported variant";
    case YK_ERR_NOMEM: return "out of memory";
    default: return "unknown";
    }
}
extern "C" const char* yk_last_cuda_error(void) { return g_lastCuda.c_str(); }

extern "C" int yk_device_count(int* count) {
    if (!count) return YK_ERR_ARG;
    *count = 0;
    CK(cudaGetDeviceCount(count));
    return YK_OK;
}

extern "C" void* yk_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void yk_host_free(void* p) { if (p) cudaFreeHost(p); }

// look-back words of yk_k_r1_offsets: one per unit of YK_R1_UNIT blocks of the (8-aligned, possibly one block larger) bound box, + ticket
static size_t r1_status_words(int W, int H) { return ((size_t)(W / 8 + 1) * (H / 8 + 1) + YK_R1_UNIT - 1) / YK_R1_UNIT + 2; }

template <class T> static int dev_alloc(YkSlotHost& s, T** out, size_t count) {
    void* p = nullptr;
    CK(cudaMalloc(&p, (count ? count : 1) * sizeof(T) + 64));
    s.devAllocs.push_back(p);
    *out = (T*)p;
    return YK_OK;
}

// TMA descriptor of one int32 plane [h][w] with a boxW x boxH box (yk_k_analyze stages regions with it).
static int encode_plane_tmap(YkTmap* tm, const void* plane, int elemBytes, size_t pitchElems, int w, int h, int boxW, int boxH) {
#ifdef YK_EMULATE
    memset(tm, 0, sizeof *tm);
    tm->opaque[0] = (unsigned long long)(uintptr_t)plane; tm->opaque[1] = (unsigned long long)w; tm->opaque[2] = (unsigned long long)h;
    tm->opaque[3] = (unsigned long long)elemBytes; tm->opaque[4] = (unsigned long long)pitchElems;
    (void)boxW; (void)boxH;
    return YK_OK;
#else
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) { g_lastCuda = "cuTensorMapEncodeTiled not available in this driver"; return YK_ERR_CUDA; }
        encode = (EncodeFn)fn;
    }
    static_assert(sizeof(YkTmap) == sizeof(CUtensorMap), "YkTmap must be a CUtensorMap");
    const cuuint64_t dims[2] = { (cuuint64_t)w, (cuuint64_t)h };
    const cuuint64_t strides[1] = { (cuuint64_t)pitchElems * (cuuint64_t)elemBytes };
    const cuuint32_t box[2] = { (cuuint32_t)boxW, (cuuint32_t)boxH };
    const cuuint32_t estr[2] = { 1, 1 };
    const CUresult r = encode(reinterpret_cast<CUtensorMap*>(tm), elemBytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_INT32, 2, (void*)plane, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_lastCuda = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r); return YK_ERR_CUDA; }
    return YK_OK;
#endif
}

static int encode_slot_tmaps(YkSlotHost& s) {
    for (int p = 0; p < s.d.nPlanes; p++) {
        const int rc = s.d.isU8
            ? encode_plane_tmap(&s.d.tmap[p], s.d.planeU8[p], 1, (size_t)s.d.pitchU8, s.d.w, s.d.h, p < 3 ? YK_U8_BOX : YK_UNIT_W, p < 3 ? YK_RAW_ROWS : 16)
            : encode_plane_tmap(&s.d.tmap[p], s.d.plane[p], 4, (size_t)s.d.w, s.d.w, s.d.h, p < 3 ? YK_RAW_PITCH : YK_UNIT_W, p < 3 ? YK_RAW_ROWS : 16);
        if (rc) return rc;
    }
    return YK_OK;
}

static int create_fill(yk_ctx* c);
extern "C" void yk_destroy(yk_ctx* c);

extern "C" int yk_create(yk_ctx** out, int device, int maxW, int maxH, int maxPlanes, int maxSlots) {
    if (!out || maxW < 4 || maxH < 4 || (maxW & 3) || (maxH & 3) || maxPlanes < 3 || maxPlanes > 4 || maxSlots < 1) return YK_ERR_ARG;
    if (maxW > 32764 || maxH > 32764) return YK_ERR_ARG;      // BoundingBox is s16 in the stream headers (YAIK_private.h:15-20)
    int n = 0;
    CK(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return YK_ERR_ARG;
    CK(cudaSetDevice(device));
    yk_ctx* c = new yk_ctx();
    c->device = device; c->maxW = maxW; c->maxH = maxH; c->maxPlanes = maxPlanes; c->maxSlots = maxSlots;
    c->slots.resize(maxSlots);
    const int rcCreate = create_fill(c);
    if (rcCreate) { yk_destroy(c); return rcCreate; }        // releases the stream and every allocation made so far
    *out = c;
    return YK_OK;
}

static int create_fill(yk_ctx* c) {
    const int maxW = c->maxW, maxH = c->maxH, maxPlanes = c->maxPlanes, maxSlots = c->maxSlots;
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    c->ownStream = true;
    { const int e = yk_analyze_setup(&c->numSMs); if (e) { g_lastCuda = std::string("yk_analyze_setup: ") + cudaGetErrorString((cudaError_t)e); return YK_ERR_CUDA; } }
    { int e = yk_preload_analyze(); if (!e) e = yk_preload_emit(); if (!e) e = yk_preload_aux();
      if (e) { g_lastCuda = std::string("kernel preload: ") + cudaGetErrorString((cudaError_t)e); return YK_ERR_CUDA; } }
    // CTAs of the persistent analysis kernel (default: one per SM).  Leaving a few SMs free lets the small ownership /
    // emission kernels of another stream run beside it when textures are pipelined over several contexts.
    c->analysisCtas = c->numSMs;
    CK(cudaMalloc((void**)&c->slotsDev, sizeof(YkSlotDev) * maxSlots));
    const size_t W = maxW, H = maxH;
    const size_t nbx = (W + 63) / 64, latW = W / 4 + 1, latH = H / 4 + 1;
    c->planeCap = W * H;
    auto up = [](size_t v) { return (v + 255) / 256 * 256; };
    // group totals of yk_k_emit (a group: YK_EMIT_THREADS nibble words or range tiles) and their super-groups
    auto groups = [](size_t n) { return (n + YK_EMIT_THREADS - 1) / YK_EMIT_THREADS; };
    auto supers = [](size_t g) { return (g + YK_SUPER - 1) / YK_SUPER; };
    size_t offTot[YK_NPASS], offSup[YK_NPASS], off = up(YK_HD_INTS * sizeof(int));
    for (int p = 0; p < YK_NPASS; p++) {
        const YkPassGeom& g = kGeom[p];
        const size_t nGroups = groups(((W + g.bw - 1) / g.bw) * ((H + g.bh - 1) / g.bh) * (size_t)g.bits / 8);
        offTot[p] = off; off += up(nGroups * sizeof(uint32_t));
        offSup[p] = off; off += up(supers(nGroups) * sizeof(uint32_t));
    }
    size_t offNib[YK_NPASS];
    for (int p = 0; p < YK_NPASS; p++) {
        const YkPassGeom& g = kGeom[p];
        offNib[p] = off;
        off += up(((W + g.bw - 1) / g.bw) * ((H + g.bh - 1) / g.bh) * (size_t)g.bits / 2 + 16);
    }
    const size_t r2Groups = groups((W / 8) * (H / 8));
    const size_t offR2Tot = off; off += up(r2Groups * sizeof(unsigned long long));
    const size_t offR2Sup = off; off += up(supers(r2Groups) * sizeof(unsigned long long));
    c->zeroABytes = off;
    const size_t offCell = off; off += up((H / 4 + 1) * nbx * sizeof(uint16_t) + 4);
    const size_t offTouch = off; off += up(latW * latH * sizeof(uint32_t));
    size_t offBitmap[YK_NPASS];          // accept bits are OR-ed in by yk_k_analyze: zero before the first pass of an image
    for (int p = 0; p < YK_NPASS; p++) {
        const YkPassGeom& g = kGeom[p];
        offBitmap[p] = off;
        off += up(((W + g.bw - 1) / g.bw) * ((H + g.bh - 1) / g.bh) * (size_t)g.bits / 8 + 8);
    }
    c->zeroStride = off;
    CK(cudaMalloc((void**)&c->zeroArea, c->zeroStride * maxSlots));
    CK(cudaMemsetAsync(c->zeroArea, 0, c->zeroStride * maxSlots, c->stream));     // on the context's own (non-blocking) stream: ordered before its first launch
    for (int i = 0; i < maxSlots; i++) {
        YkSlotHost& s = c->slots[i];
        memset(&s.d, 0, sizeof s.d);
        int rc;
        uint8_t* za = c->zeroArea + c->zeroStride * i;
        for (int p = 0; p < maxPlanes; p++) if ((rc = dev_alloc(s, &s.owned[p], W * H))) return rc;
        for (int p = 0; p < maxPlanes; p++) if ((rc = dev_alloc(s, &s.ownedU8[p], ((W + 15) / 16 * 16) * H + 256))) return rc;
        s.d.hdr = (int*)za;
        for (int p = 0; p < YK_NPASS; p++) { s.d.rgbTot[p] = (uint32_t*)(za + offTot[p]); s.d.rgbSup[p] = (uint32_t*)(za + offSup[p]); }
        for (int p = 0; p < YK_NPASS; p++) s.d.emitNib[p] = (uint32_t*)(za + offNib[p]);
        s.d.r2Tot = (unsigned long long*)(za + offR2Tot);
        s.d.r2Sup = (unsigned long long*)(za + offR2Sup);
        s.d.cellMask = (uint16_t*)(za + offCell);
        s.d.touchMap = (uint32_t*)(za + offTouch);
        if ((rc = dev_alloc(s, &s.d.alphaKept, ((H + 15) / 16) * ((W + 15) / 16)))) return rc;
        for (int p = 0; p < YK_NPASS; p++) {
            const YkPassGeom& g = kGeom[p];
            s.d.bitmap[p] = za + offBitmap[p];
            if ((rc = dev_alloc(s, &s.d.rgb[p], 3 * ((W >> g.shx) + 1) * ((H >> g.shy) + 1)))) return rc;
        }
        if ((rc = dev_alloc(s, &s.d.latRGB, latW * latH * 3))) return rc;
        for (int p = 0; p < 3; p++) {
            if ((rc = dev_alloc(s, &s.d.r2Raw[p], W * H + 64))) return rc;
            if ((rc = dev_alloc(s, &s.d.r2RawType[p], (W / 8 + 1) * (H / 8 + 1)))) return rc;
            if ((rc = dev_alloc(s, &s.d.r2Idx[p], W * H))) return rc;
            if ((rc = dev_alloc(s, &s.d.r2Type[p], 3 * (W / 8 + 1) * (H / 8 + 1)))) return rc;
        }
        if ((rc = dev_alloc(s, &s.d.r1Status, r1_status_words(W, H)))) return rc;
        { uint4* list = nullptr; if ((rc = dev_alloc(s, &list, (W / 8 + 1) * (H / 8 + 1) + 1))) return rc; s.d.r1List = list; }
        for (int p = 0; p < 3; p++) {
            if ((rc = dev_alloc(s, &s.d.r1Nib[p], (W / 8) * (H / 8) * 8 + 4))) return rc;
            if ((rc = dev_alloc(s, &s.d.r1Defs[p], (W / 8) * (H / 8) + 4))) return rc;
        }
    }
    { const char* e = getenv("YK_PACK_THREADS"); c->packer = yk_hostpack_create(e ? atoi(e) : 0); }
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}

extern "C" void yk_destroy(yk_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->ownStream || c->stream) cudaStreamSynchronize(c->stream);
    for (auto& s : c->slots) {
        for (void* p : s.devAllocs) cudaFree(p);
        if (s.haloIn) cudaFree(s.haloIn);
        if (s.stageHost) cudaFreeHost(s.stageHost);
        if (s.arena) cudaFreeHost(s.arena);
        if (s.stageFree) cudaEventDestroy(s.stageFree);
    }
    if (c->packer) yk_hostpack_destroy(c->packer);
    cudaFree(c->slotsDev); cudaFree(c->zeroArea);
    if (c->stage8) cudaFree(c->stage8);
    if (c->lutDev) cudaFree(c->lutDev);
    if (c->rtabDev) cudaFree(c->rtabDev);
    if (c->r7Dev) cudaFree(c->r7Dev);
    if (c->ownStream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int yk_set_stream(yk_ctx* c, void* st) {
    if (!c) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    if (c->ownStream) { cudaStreamDestroy(c->stream); c->ownStream = false; }
    c->stream = (cudaStream_t)st;
    return YK_OK;
}
extern "C" int yk_sync(yk_ctx* c) {
    if (!c) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}
extern "C" long long yk_launch_count(yk_ctx* c) { return c ? c->launches : 0; }

extern "C" int yk_set_analysis_ctas(yk_ctx* c, int ctas) {
    if (!c || ctas < 0) return YK_ERR_ARG;
    c->analysisCtas = (ctas == 0 || ctas > c->numSMs) ? c->numSMs : ctas;
    return YK_OK;
}
extern "C" int yk_sm_count(yk_ctx* c) { return c ? c->numSMs : 0; }

extern "C" int yk_profile(yk_ctx* c, int enable) {
    if (!c) return YK_ERR_ARG;
    c->profile = enable != 0;
    return YK_OK;
}
extern "C" int yk_profile_read(yk_ctx* c, double ms[8], long long count[8]) {
    if (!c || !ms || !count) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    for (int k = 0; k < 8; k++) { ms[k] = 0; count[k] = 0; }
    for (int k = 0; k < 6; k++) {
        for (size_t i = 0; i < c->evA[k].size(); i++) {
            float t = 0;
            if (cudaEventElapsedTime(&t, c->evA[k][i], c->evB[k][i]) == cudaSuccess) { ms[k] += t; count[k]++; }
            cudaEventDestroy(c->evA[k][i]); cudaEventDestroy(c->evB[k][i]);
        }
        c->evA[k].clear(); c->evB[k].clear();
    }
    return YK_OK;
}

static int slot_ok(yk_ctx* c, int slot) { return c && slot >= 0 && slot < c->maxSlots; }
static int upload_slots_fwd(yk_ctx* c, int slot0, int nSlots);

static int configure_slot(yk_ctx* c, int slot, int nPlanes, int w, int h) {
    if (nPlanes < 3 || nPlanes > 4 || w < 4 || h < 4 || (w & 3) || (h & 3)) return YK_ERR_ARG;
    if (w > c->maxW || h > c->maxH || (size_t)w * h > c->planeCap || nPlanes > c->maxPlanes) return YK_ERR_CAPACITY;
    YkSlotHost& s = c->slots[slot];
    s.d.w = w; s.d.h = h; s.d.nPlanes = nPlanes;
    s.d.nbx = (w + 63) / 64; s.d.nby = (h + 63) / 64;
    s.d.imgH = h; s.d.y0 = 0; s.d.hasAbove = 0; s.d.hasBelow = 0; s.d.touchInTop = nullptr; s.d.touchInBottom = nullptr;
    s.d.latW = w / 4 + 1; s.d.latH = h / 4 + 1;
    for (int p = 0; p < 3; p++) s.d.rowBelow[p] = nullptr;
    s.haveImage = true; s.dirty = true; s.chromaReady = false; s.strip = false;
    return YK_OK;
}

static void mark_reset(YkSlotHost& s) {
    s.zeroAClean = true; s.touchDirty = false; s.cellsClean = true; s.harvested = false;
    if (s.d.alphaReset || s.d.alphaValid) s.dirty = true;
    s.d.alphaReset = 0; s.d.alphaValid = 0;
    s.k1Ran = s.alphaRan = s.alphaFetched = s.prepared = s.r2Valid = s.pendingHarvest = false;
    s.r1Fused = 0; s.r1Strip = 0;
    s.nextPass = 0; s.rangeErr = 0; s.lastRunPasses = 0;
    memset(s.hdr, 0, sizeof s.hdr);
}

extern "C" int yk_reset_state(yk_ctx* c, int slot) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    CK(cudaMemsetAsync(c->zeroArea + c->zeroStride * slot, 0, c->zeroStride, c->stream));
    mark_reset(s);
    return YK_OK;
}

// the same for slots [slot0, slot0 + nSlots) with one clear (their state areas are contiguous)
extern "C" int yk_reset_states(yk_ctx* c, int slot0, int nSlots) {
    if (!c || nSlots < 1 || slot0 < 0 || slot0 + nSlots > c->maxSlots) return YK_ERR_ARG;
    for (int i = slot0; i < slot0 + nSlots; i++) if (!c->slots[i].haveImage) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    CK(cudaMemsetAsync(c->zeroArea + c->zeroStride * slot0, 0, c->zeroStride * nSlots, c->stream));
    for (int i = slot0; i < slot0 + nSlots; i++) mark_reset(c->slots[i]);
    return YK_OK;
}

extern "C" int yk_set_upload_format(yk_ctx* c, int packedU8) {
    if (!c) return YK_ERR_ARG;
    c->packedUpload = packedU8 != 0;
    return YK_OK;
}

// The slot's samples are in its own packed planes (ownedU8, row pitch (w + 15) / 16 * 16, padding zero): the state every
// stage expects after a packed upload, whichever way the bytes arrived.
static int use_packed_planes(yk_ctx* c, int slot) {
    YkSlotHost& s = c->slots[slot];
    for (int p = 0; p < 4; p++) {
        s.d.planeU8[p] = p < s.d.nPlanes ? s.ownedU8[p] : nullptr;
        s.d.plane[p] = p < s.d.nPlanes ? s.owned[p] : nullptr;
    }
    s.d.isU8 = 1; s.d.pitchU8 = (s.d.w + 15) / 16 * 16;
    s.int32Valid = false;
    s.borrowed = false;
    const int rc = encode_slot_tmaps(s);
    if (rc) return rc;
    return yk_reset_state(c, slot);
}

extern "C" int yk_set_image(yk_ctx* c, int slot, const int32_t* const* planes, int nPlanes, int w, int h) {
    if (!slot_ok(c, slot) || !planes) return YK_ERR_ARG;
    int rc = configure_slot(c, slot, nPlanes, w, h);
    if (rc) return rc;
    YkSlotHost& s = c->slots[slot];
    CK(cudaSetDevice(c->device));
    for (int p = 0; p < nPlanes; p++) if (!planes[p]) return YK_ERR_ARG;
    unsigned bad = 0;
    if (c->packedUpload) {
        // Plane samples are 0..255 on this path: pack them to bytes on the host (threads, range check included) and move a
        // quarter of the bytes over PCIe; yk_k_analyze_u8 stages the packed planes with byte TMA boxes
        const size_t pitch = ((size_t)w + 15) / 16 * 16, planeBytes = pitch * h, need = planeBytes * nPlanes;
        if (s.stageBytes < need) {
            if (s.stageBusy) { CK(cudaEventSynchronize(s.stageFree)); s.stageBusy = false; }
            if (s.stageHost) cudaFreeHost(s.stageHost);
            s.stageHost = nullptr; s.stageBytes = 0;
            CK(cudaMallocHost((void**)&s.stageHost, need));
            s.stageBytes = need;
        }
        if (!s.stageFree) CK(cudaEventCreateWithFlags(&s.stageFree, cudaEventDisableTiming));
        if (s.stageBusy) { CK(cudaEventSynchronize(s.stageFree)); s.stageBusy = false; }     // the previous upload has left the staging buffer
        for (int p = 0; p < nPlanes; p++) {
            bad |= yk_hostpack_plane(c->packer, planes[p], s.stageHost + p * planeBytes, w, h, pitch);
            CK(cudaMemcpyAsync(s.ownedU8[p], s.stageHost + p * planeBytes, planeBytes, cudaMemcpyHostToDevice, c->stream));      // overlaps the packing of the next plane
        }
        CK(cudaEventRecord(s.stageFree, c->stream));
        s.stageBusy = true;
        if (!(bad & ~255u)) return use_packed_planes(c, slot);
        // samples outside 0..255 (signed chroma planes): this image goes up as int32 instead.  yk_range_dyn takes such
        // planes; the alpha / gradient / 1-D range stages report YK_ERR_RANGE for them either way.
    }
    for (int p = 0; p < nPlanes; p++) {
        CK(cudaMemcpyAsync(s.owned[p], planes[p], (size_t)w * h * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        s.d.plane[p] = s.owned[p];
        s.d.planeU8[p] = nullptr;
    }
    s.d.isU8 = 0; s.d.pitchU8 = 0;
    s.int32Valid = true;
    for (int p = nPlanes; p < 4; p++) { s.d.plane[p] = nullptr; s.d.planeU8[p] = nullptr; }
    s.borrowed = false;
    if ((rc = encode_slot_tmaps(s))) return rc;
    rc = yk_reset_state(c, slot);
    if (bad & ~255u) s.rangeErr = 1;
    return rc;
}

// the kernels outside the hot path (state download, DynamicTileEncode) read Plane-style int32 samples
static int ensure_int32(yk_ctx* c, int slot) {
    YkSlotHost& s = c->slots[slot];
    if (s.int32Valid) return YK_OK;
    int rc = upload_slots_fwd(c, slot, 1);
    if (rc) return rc;
    yk_launch_expand(c->slotsDev, slot, s.d.nPlanes, s.d.w, s.d.h, s.owned, c->stream);
    c->launches++;
    CK(cudaGetLastError());
    s.int32Valid = true;
    return YK_OK;
}

extern "C" int yk_set_image_device(yk_ctx* c, int slot, const int32_t* const* devPlanes, int nPlanes, int w, int h) {
    if (!slot_ok(c, slot) || !devPlanes) return YK_ERR_ARG;
    int rc = configure_slot(c, slot, nPlanes, w, h);
    if (rc) return rc;
    YkSlotHost& s = c->slots[slot];
    for (int p = 0; p < nPlanes; p++) {
        if (!devPlanes[p] || ((uintptr_t)devPlanes[p] & 15)) return YK_ERR_ARG;
        s.d.plane[p] = devPlanes[p];
        s.d.planeU8[p] = nullptr;
    }
    s.d.isU8 = 0; s.d.pitchU8 = 0; s.int32Valid = true;
    for (int p = nPlanes; p < 4; p++) s.d.plane[p] = nullptr;
    s.borrowed = true;
    if ((rc = encode_slot_tmaps(s))) return rc;
    return yk_reset_state(c, slot);
}

// Interleaved 8-bit pixels at `src` (device memory, or the context's staging copy) into the slot's packed planes
static int unpack_interleaved(yk_ctx* c, int slot, const uint8_t* src, size_t rowBytes, int channels) {
    YkSlotHost& s = c->slots[slot];
    YkUnpackArgs a;
    a.src = src; a.rowBytes = rowBytes; a.nPlanes = s.d.nPlanes; a.w = s.d.w; a.h = s.d.h; a.pitch = (s.d.w + 15) / 16 * 16;
    for (int p = 0; p < 4; p++) a.dst[p] = p < s.d.nPlanes ? s.ownedU8[p] : nullptr;
    { YkTimed t(c, 5); yk_launch_unpack8(a, channels, c->stream); }
    c->launches++;
    CK(cudaGetLastError());
    return use_packed_planes(c, slot);
}

static int check_interleaved(yk_ctx* c, int slot, const uint8_t* pixels, size_t rowBytes, int channels, int nPlanes, int w, int h) {
    if (!slot_ok(c, slot) || !pixels || (channels != 3 && channels != 4) || (nPlanes != 3 && nPlanes != channels)) return YK_ERR_ARG;
    if (w < 0 || rowBytes < (size_t)w * channels) return YK_ERR_ARG;
    return configure_slot(c, slot, nPlanes, w, h);
}

extern "C" int yk_set_image_interleaved(yk_ctx* c, int slot, const uint8_t* pixels, size_t rowBytes, int channels, int nPlanes, int w, int h) {
    int rc = check_interleaved(c, slot, pixels, rowBytes, channels, nPlanes, w, h);
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    // one copy of the span from the first pixel to the last pixel's last byte, never past it (a decoder's buffer often ends there)
    const size_t need = rowBytes * (h - 1) + (size_t)w * channels;
    if (c->stage8Bytes < need) {
        if (c->stage8) { CK(cudaStreamSynchronize(c->stream)); cudaFree(c->stage8); }
        c->stage8 = nullptr; c->stage8Bytes = 0;
        CK(cudaMalloc((void**)&c->stage8, need));
        c->stage8Bytes = need;
    }
    CK(cudaMemcpyAsync(c->stage8, pixels, need, cudaMemcpyHostToDevice, c->stream));
    return unpack_interleaved(c, slot, c->stage8, rowBytes, channels);
}

extern "C" int yk_set_image_interleaved_device(yk_ctx* c, int slot, const uint8_t* devPixels, size_t rowBytes, int channels, int nPlanes, int w, int h) {
    int rc = check_interleaved(c, slot, devPixels, rowBytes, channels, nPlanes, w, h);
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    return unpack_interleaved(c, slot, devPixels, rowBytes, channels);
}

extern "C" int32_t* yk_device_plane(yk_ctx* c, int slot, int p) {
    if (!slot_ok(c, slot) || p < 0 || p >= c->maxPlanes) return nullptr;
    return c->slots[slot].owned[p];
}

static int upload_slots(yk_ctx* c, int slot0, int nSlots);
static int upload_slots_fwd(yk_ctx* c, int slot0, int nSlots) { return upload_slots(c, slot0, nSlots); }
static int upload_slots(yk_ctx* c, int slot0, int nSlots) {
    for (int i = slot0; i < slot0 + nSlots; i++) {
        YkSlotHost& s = c->slots[i];
        if (s.dirty) {
            if (c->noHostWait) return YK_ERR_STATE;
            CK(cudaMemcpyAsync(c->slotsDev + i, &s.d, sizeof(YkSlotDev), cudaMemcpyHostToDevice, c->stream));
            s.dirty = false;
        }
    }
    return YK_OK;
}

static int check_batch(yk_ctx* c, int slot0, int nSlots) {
    if (!c || nSlots < 1 || slot0 < 0 || slot0 + nSlots > c->maxSlots) return YK_ERR_ARG;
    const YkSlotHost& a = c->slots[slot0];
    for (int i = slot0; i < slot0 + nSlots; i++) {
        const YkSlotHost& s = c->slots[i];
        if (!s.haveImage) return YK_ERR_STATE;
        if (s.d.w != a.d.w || s.d.h != a.d.h || s.d.isU8 != a.d.isU8) return YK_ERR_ARG;
    }
    return YK_OK;
}

// Copy back the header of the last run (one sync) and keep what that run produced: the stats of its passes, the
// alpha box if it ran the alpha stage, the R2 totals (the scan always refreshes them).
static int fetch_hdr(yk_ctx* c, YkSlotHost& s) {
    if (s.pendingHarvest) {
        if (c->noHostWait) return YK_ERR_STATE;
        int tmp[YK_HD_INTS];
        CK(cudaMemcpyAsync(tmp, s.d.hdr, sizeof tmp, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        s.pendingHarvest = false;
        if (tmp[YK_HD_ERR] & 1) s.rangeErr = 1;
        for (int p = 0; p < YK_NPASS; p++)
            if (s.lastRunPasses & (1 << p)) memcpy(s.hdr + YK_HD_PASS0 + p * YK_ST_STRIDE, tmp + YK_HD_PASS0 + p * YK_ST_STRIDE, YK_ST_STRIDE * sizeof(int));
        if (s.lastRunPasses & 256) memcpy(s.hdr + YK_HD_ALPHA_KEPT0, tmp + YK_HD_ALPHA_KEPT0, 5 * sizeof(int));
        s.hdr[YK_HD_R2_CHUNKS] = tmp[YK_HD_R2_CHUNKS]; s.hdr[YK_HD_R2_TILES] = tmp[YK_HD_R2_TILES];
    }
    return s.rangeErr ? YK_ERR_RANGE : YK_OK;
}

// Enqueue analysis kernels for a run (list of gradient passes, optional alpha), then the emission + scan + R2 tail.
static int enqueue(yk_ctx* c, int slot0, int nSlots, const YkRun& run, bool doEmit, bool doR2, int phases = 3) {
    int rc = check_batch(c, slot0, nSlots);
    if (rc) return rc;
    for (int p = 1; p < run.nPasses; p++) if (run.passId[p] <= run.passId[p - 1]) return YK_ERR_ARG;   // the kernel runs a launch's passes in Convert()'s order
    CK(cudaSetDevice(c->device));
    const YkSlotHost& a = c->slots[slot0];
    const int nRegions = a.d.nbx * a.d.nby;
    for (int i = slot0; i < slot0 + nSlots && (phases & 1); i++)            // the header is about to be cleared: keep the previous run's numbers
        if (c->slots[i].pendingHarvest) { rc = fetch_hdr(c, c->slots[i]); if (rc && rc != YK_ERR_RANGE) return rc; }
    bool needFold = false;
    for (int i = slot0; i < slot0 + nSlots && (phases & 1); i++) {
        YkSlotHost& s = c->slots[i];
        if (!s.zeroAClean) CK(cudaMemsetAsync(c->zeroArea + c->zeroStride * i, 0, c->zeroABytes, c->stream));
        s.zeroAClean = false;
        if (s.touchDirty && run.nPasses > 0) needFold = true;
    }
    bool fresh = true;
    for (int i = slot0; i < slot0 + nSlots && (phases & 1); i++) {
        YkSlotHost& s = c->slots[i];
        if (!s.cellsClean) {
            fresh = false;
            // a pass that runs again on a used state starts from an empty bitmap (FittingQuadSmooth allocates pFillBitMap per call, EC.cpp:3770-3777)
            for (int p = 0; p < run.nPasses; p++) {
                const YkPassGeom& g = kGeom[run.passId[p]];
                const size_t nb = (size_t)((s.d.w + g.bw - 1) / g.bw) * ((s.d.h + g.bh - 1) / g.bh) * g.bits / 8;
                CK(cudaMemsetAsync(s.d.bitmap[run.passId[p]], 0, nb, c->stream));
            }
        }
    }
    if ((rc = upload_slots(c, slot0, nSlots))) return rc;
    if (needFold) { yk_launch_fold_touch(c->slotsDev, slot0, nSlots, a.d.latW * a.d.latH, c->stream); c->launches++; }
    const bool r2Domain = doR2 && !(a.d.w & 7) && !(a.d.h & 7);
    YkRun krun = run;
    krun.doR2 = r2Domain ? 1 : 0;
    krun.fresh = fresh ? 1 : 0;
    // a launch that has the GPU to itself balances its tail by taking its last units on demand; a partial launch runs
    // beside others (pipelined contexts) which fill its tail anyway
    krun.endgameUnits = c->analysisCtas >= c->numSMs ? YK_ENDGAME_UNITS : 0;
    if ((phases & 1) && (krun.nPasses > 0 || krun.doAlpha || krun.doR2)) {
        YkTimed t(c, 0);
        yk_launch_analyze(c->slotsDev, slot0, nSlots, nRegions, c->analysisCtas, a.d.isU8 != 0, krun, c->stream); c->launches++;
    }
    if (phases & 2) {
        // ownership of the touched lattice points, then one scan/compaction kernel: rgbStream emission of the run's
        // passes + gather of the range stage's per-tile output into stream order
        int gradGroups = 0;
        if (doEmit)
            for (int p = 0; p < krun.nPasses; p++) {
                const YkPassGeom& g = kGeom[krun.passId[p]];
                const int nWords = ((a.d.w + g.bw - 1) / g.bw) * ((a.d.h + g.bh - 1) / g.bh) * g.bits / 8;
                gradGroups += (nWords + YK_EMIT_THREADS - 1) / YK_EMIT_THREADS;
            }
        const int nTiles = (a.d.w / 8) * (a.d.h / 8);
        const int r2Groups = (r2Domain && nTiles > 0) ? (nTiles + YK_EMIT_THREADS - 1) / YK_EMIT_THREADS : 0;
        if (gradGroups + r2Groups > 0) { YkTimed t(c, 2); yk_launch_owner(c->slotsDev, slot0, nSlots, a.d.latW * a.d.latH, gradGroups > 0, krun, c->stream); c->launches++; }
        if (gradGroups + r2Groups > 0) { YkTimed t(c, 1); yk_launch_emit(c->slotsDev, slot0, nSlots, gradGroups, r2Groups, krun, c->stream); c->launches++; }
    }
    CK(cudaGetLastError());
    for (int i = slot0; i < slot0 + nSlots; i++) {
        YkSlotHost& s = c->slots[i];
        s.k1Ran = true; s.pendingHarvest = true; s.harvested = false; s.lastRunPasses = (run.doAlpha ? 256 : 0);
        if (run.nPasses > 0 || run.doAlpha) s.r1Fused = 0;       // the masks DynamicTileEncode works on are changing
        for (int p = 0; p < run.nPasses; p++) s.lastRunPasses |= 1 << run.passId[p];
        if (run.doAlpha && s.d.nPlanes == 4) { s.alphaRan = true; s.alphaFetched = false; }
        if (run.nPasses > 0) { s.r2Valid = false; s.touchDirty = true; s.cellsClean = false; }
        if (doR2) s.r2Valid = true;
    }
    return YK_OK;
}

static int enqueue_r1_fused(yk_ctx* c, int slot, int mode3BitOnly, bool useAlpha);

extern "C" int yk_analyze(yk_ctx* c, int slot0, int nSlots, int stages, int rejectFactor) {
    if (!c || rejectFactor < 0 || rejectFactor > 64) return YK_ERR_ARG;
    if ((stages & YK_STAGE_RANGEDYN) && (stages & YK_STAGE_RANGEDYN3)) return YK_ERR_ARG;
    YkRun run; memset(&run, 0, sizeof run);
    run.rejectFactor = rejectFactor;
    run.doAlpha = (stages & YK_STAGE_ALPHA) ? 1 : 0;
    if (stages & YK_STAGE_GRADIENT) { run.nPasses = YK_NPASS; for (int i = 0; i < YK_NPASS; i++) run.passId[i] = i; }
    int rc = check_batch(c, slot0, nSlots);
    if (rc) return rc;
    if (stages & YK_STAGE_GRADIENT)
        for (int i = slot0; i < slot0 + nSlots; i++) if (c->slots[i].prepared || c->slots[i].nextPass) return YK_ERR_STATE;   // needs a fresh state
    rc = enqueue(c, slot0, nSlots, run, true, (stages & YK_STAGE_RANGE1D) != 0);
    if (rc) return rc;
    if (stages & YK_STAGE_GRADIENT)
        for (int i = slot0; i < slot0 + nSlots; i++) { c->slots[i].prepared = true; c->slots[i].preparedReject = rejectFactor; c->slots[i].nextPass = 0; }
    if (stages & (YK_STAGE_RANGEDYN | YK_STAGE_RANGEDYN3))
        for (int i = slot0; i < slot0 + nSlots; i++) {
            const YkSlotHost& s = c->slots[i];
            // the alpha box the coder works in: of this run, or (host-side flags) of an earlier yk_alpha_reject
            const bool alphaThisRun = (stages & YK_STAGE_ALPHA) && s.d.nPlanes == 4;
            if (!alphaThisRun && s.alphaRan) return YK_ERR_STATE;       // an earlier alpha stage: code the planes with yk_range_dyn
            if ((rc = enqueue_r1_fused(c, i, (stages & YK_STAGE_RANGEDYN3) != 0, alphaThisRun))) return rc;
        }
    return YK_OK;
}

extern "C" int yk_prepare_quad_smooth(yk_ctx* c, int slot, int rejectFactor) {
    return yk_analyze(c, slot, 1, YK_STAGE_GRADIENT, rejectFactor);
}

// ---- results to the host ---------------------------------------------------------------------------------
// One pinned arena per slot receives every result stream of the last run with two synchronisations (the header with the
// stream lengths first, then all streams at their actual sizes); the getters then serve from it.
static size_t pass_bitmap_bytes(const YkSlotHost& s, int p) {
    const YkPassGeom& g = kGeom[p];
    return (size_t)((s.d.w + g.bw - 1) / g.bw) * ((s.d.h + g.bh - 1) / g.bh) * g.bits / 8;
}
static int harvest(yk_ctx* c, YkSlotHost& s) {
    if (s.harvested) return s.rangeErr ? YK_ERR_RANGE : YK_OK;
    int rc = fetch_hdr(c, s);
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    const int mask = s.prepared ? (1 << YK_NPASS) - 1 : (s.lastRunPasses & ((1 << YK_NPASS) - 1));
    auto up = [](size_t v) { return (v + 63) / 64 * 64; };
    size_t off = 0;
    for (int p = 0; p < YK_NPASS; p++) {
        s.arBitmap[p] = off; if (mask & (1 << p)) off += up(pass_bitmap_bytes(s, p));
        s.arRgb[p] = off; if (mask & (1 << p)) off += up((size_t)s.hdr[YK_HD_PASS0 + p * YK_ST_STRIDE + YK_ST_RGBBYTES]);
    }
    const size_t ni = 16ull * (size_t)s.hdr[YK_HD_R2_CHUNKS], nt = 3ull * (size_t)s.hdr[YK_HD_R2_TILES];
    for (int pl = 0; pl < 3; pl++) {
        s.arIdx[pl] = off; if (s.r2Valid) off += up(ni);
        s.arType[pl] = off; if (s.r2Valid) off += up(nt);
    }
    const bool wantKept = s.alphaRan && s.d.nPlanes == 4;
    const size_t nKept = (size_t)((s.d.w + 15) / 16) * ((s.d.h + 15) / 16);
    s.arKept = off; if (wantKept) off += up(nKept);
    if (off > s.arenaBytes) {
        if (s.arena) cudaFreeHost(s.arena);
        s.arena = nullptr; s.arenaBytes = 0;
        const size_t want = off + off / 4 + 4096;
        CK(cudaMallocHost((void**)&s.arena, want));
        s.arenaBytes = want;
    }
    for (int p = 0; p < YK_NPASS; p++) {
        if (!(mask & (1 << p))) continue;
        CK(cudaMemcpyAsync(s.arena + s.arBitmap[p], s.d.bitmap[p], pass_bitmap_bytes(s, p), cudaMemcpyDeviceToHost, c->stream));
        const size_t nrgb = (size_t)s.hdr[YK_HD_PASS0 + p * YK_ST_STRIDE + YK_ST_RGBBYTES];
        if (nrgb) CK(cudaMemcpyAsync(s.arena + s.arRgb[p], s.d.rgb[p], nrgb, cudaMemcpyDeviceToHost, c->stream));
    }
    if (s.r2Valid)
        for (int pl = 0; pl < 3; pl++) {
            if (ni) CK(cudaMemcpyAsync(s.arena + s.arIdx[pl], s.d.r2Idx[pl], ni, cudaMemcpyDeviceToHost, c->stream));
            if (nt) CK(cudaMemcpyAsync(s.arena + s.arType[pl], s.d.r2Type[pl], nt, cudaMemcpyDeviceToHost, c->stream));
        }
    if (wantKept) CK(cudaMemcpyAsync(s.arena + s.arKept, s.d.alphaKept, nKept, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    s.arMask = mask; s.arR2 = s.r2Valid; s.arHasKept = wantKept;
    s.harvested = true;
    return YK_OK;
}

// ---- alpha ------------------------------------------------------------------------------------------------
static int alpha_finish(yk_ctx* c, YkSlotHost& s) {
    if (s.alphaFetched) return YK_OK;
    int rc = fetch_hdr(c, s);
    if (rc) return rc;
    const int w = s.d.w, h = s.d.h;
    const int tw = (w + 15) / 16, th = (h + 15) / 16;
    if (!yk_alpha_box(s.hdr, w, s.bound)) return YK_ERR_ARG;     // fully transparent: outside the reference's domain (sentinel bbox)
    const int L = s.bound[0], T = s.bound[1], R = s.bound[2], B = s.bound[3];
    s.alphaBitmap.clear();
    if (!yk_box_is_image(s.bound, w, s.d.imgH)) {
        std::vector<uint8_t> keptBuf;
        const uint8_t* kept;
        if (s.harvested && s.arHasKept) kept = s.arena + s.arKept;
        else {
            keptBuf.resize((size_t)tw * th);
            CK(cudaMemcpyAsync(keptBuf.data(), s.d.alphaKept, keptBuf.size(), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            kept = keptBuf.data();
        }
        const int bx0 = L >> 4, bx1 = (R + 15) >> 4, by0 = T >> 4, by1 = (B + 15) >> 4;
        const int tWB = bx1 - bx0, tHB = by1 - by0;
        s.alphaBitmap.assign((size_t)(tWB * tHB + 7) / 8, 0);
        int bit = 0, rem = 0;
        for (int y = 0; y < tHB; y++)
            for (int x = 0; x < tWB; x++, bit++)
                if (kept[(size_t)(y + by0) * tw + x + bx0]) { s.alphaBitmap[bit >> 3] |= (uint8_t)(1 << (bit & 7)); rem += 256; }   // EC.cpp:1317-1327
        s.remaining = rem; s.wroteChunk = 1;
        s.chunkBBox[0] = bx0; s.chunkBBox[1] = by0; s.chunkBBox[2] = tWB; s.chunkBBox[3] = tHB;
        s.d.alphaReset = 0;
    } else {
        s.remaining = R * B; s.wroteChunk = 0; s.d.alphaReset = 1;     // EC.cpp:1400-1403
    }
    s.d.alphaValid = 1; s.dirty = true; s.alphaFetched = true;
    return YK_OK;
}

extern "C" int yk_alpha_reject(yk_ctx* c, int slot, uint8_t* bitmap, int bitmapCap, int* bitmapBytes, int boundPx[4],
                               int* remainingPixels, int* wroteChunk, int chunkBBoxTiles[4]) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    if (s.d.nPlanes != 4) return YK_ERR_ARG;
    if (s.d.hasAbove || s.d.hasBelow) return YK_ERR_UNSUPPORTED;    // the alpha bitmap of a strip set is not assembled here
    if (!s.alphaRan) {
        YkRun run; memset(&run, 0, sizeof run); run.doAlpha = 1; run.rejectFactor = 3;
        int rc = enqueue(c, slot, 1, run, false, false);
        if (rc) return rc;
    }
    int rc = alpha_finish(c, s);
    if (rc) return rc;
    if ((int)s.alphaBitmap.size() > bitmapCap) return YK_ERR_CAPACITY;
    if (bitmap && !s.alphaBitmap.empty()) memcpy(bitmap, s.alphaBitmap.data(), s.alphaBitmap.size());
    if (bitmapBytes) *bitmapBytes = (int)s.alphaBitmap.size();
    if (boundPx) memcpy(boundPx, s.bound, sizeof s.bound);
    if (remainingPixels) *remainingPixels = s.remaining;
    if (wroteChunk) *wroteChunk = s.wroteChunk;
    if (chunkBBoxTiles) memcpy(chunkBBoxTiles, s.chunkBBox, sizeof s.chunkBBox);
    return YK_OK;
}

// ---- gradient ---------------------------------------------------------------------------------------------
extern "C" int yk_gradient_pass(yk_ctx* c, int slot, int rejectFactor, int shX, int shY,
                                uint8_t* bitmap, int bitmapCap, int* bitmapBytes,
                                uint8_t* rgb, int rgbCap, int* rgbBytes, int bbox[4], int* tileDone) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    const int pid = pass_id(shX, shY);
    if (pid < 0 || rejectFactor < 0 || rejectFactor > 64) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    int rc;
    if (s.prepared) {
        // results of the fused cascade are only what the reference would compute if the passes are consumed in
        // Convert()'s order with the same rejectFactor
        if (pid != s.nextPass || rejectFactor != s.preparedReject) return YK_ERR_STATE;
    } else {
        YkRun run; memset(&run, 0, sizeof run);
        run.nPasses = 1; run.passId[0] = pid; run.rejectFactor = rejectFactor;
        if ((rc = enqueue(c, slot, 1, run, true, false))) return rc;
        s.nextPass = -1;
    }
    if ((rc = harvest(c, s))) return rc;
    const int w = s.d.w;
    const int nb = (int)pass_bitmap_bytes(s, pid);
    const int* st = s.hdr + YK_HD_PASS0 + pid * YK_ST_STRIDE;
    const int nrgb = st[YK_ST_RGBBYTES];
    if (nb > bitmapCap || nrgb > rgbCap) return YK_ERR_CAPACITY;
    if (bitmap) memcpy(bitmap, s.arena + s.arBitmap[pid], nb);
    if (rgb && nrgb) memcpy(rgb, s.arena + s.arRgb[pid], nrgb);
    if (s.prepared) s.nextPass++;          // consumed only now: a capacity / CUDA error above leaves the pass available for a retry
    if (bitmapBytes) *bitmapBytes = nb;
    if (rgbBytes) *rgbBytes = nrgb;
    if (tileDone) *tileDone = st[YK_ST_TILEDONE];
    if (bbox) {
        bbox[0] = w - st[YK_ST_MINX];
        bbox[1] = st[YK_ST_MINY] ? INT_MAX / 2 - st[YK_ST_MINY] : s.d.imgH;
        bbox[2] = st[YK_ST_MAXX]; bbox[3] = st[YK_ST_MAXY];
    }
    return YK_OK;
}

// ---- range R2 ---------------------------------------------------------------------------------------------
extern "C" int yk_range1d(yk_ctx* c, int slot, int plane, uint8_t* idx, int idxCap, int* idxBytes,
                          uint8_t* type, int typeCap, int* typeBytes) {
    if (!slot_ok(c, slot) || plane < 0 || plane > 2) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    if ((s.d.w & 7) || (s.d.h & 7)) return YK_ERR_ARG;          // the reference's own domain (SURVEY.md hazard 11)
    int rc;
    if (!s.r2Valid) {
        YkRun run; memset(&run, 0, sizeof run); run.rejectFactor = 3;      // no gradient pass: code the unclaimed tiles, scan, gather
        if ((rc = enqueue(c, slot, 1, run, false, true))) return rc;
    }
    if ((rc = harvest(c, s))) return rc;
    const long long ni = 16ll * s.hdr[YK_HD_R2_CHUNKS], nt = 3ll * s.hdr[YK_HD_R2_TILES];
    if (ni > idxCap || nt > typeCap) return YK_ERR_CAPACITY;
    if (idx && ni) memcpy(idx, s.arena + s.arIdx[plane], (size_t)ni);
    if (type && nt) memcpy(type, s.arena + s.arType[plane], (size_t)nt);
    if (idxBytes) *idxBytes = (int)ni;
    if (typeBytes) *typeBytes = (int)nt;
    return YK_OK;
}


// ---- range R1 ---------------------------------------------------------------------------------------------
// Six LUTs per (base6, range7) pair, built on the host with the reference's own float expression and glibc powf
// (DynamicTile::buildTable, EC.cpp:625-699; SURVEY.md hazard 12).  range7 can exceed 7 bits for bases close to 224
// (a reference quirk: EncodeTileType then spills into the type bits) — the table simply covers it.
// Behind the 72 entries sit the 72 decision thresholds yk_k_r1_encode searches with (see there): the LUTs are
// non-decreasing (checked here: the kernel's search depends on it), so "first strict minimum of |entry - value|"
// is "number of thresholds below the value".
struct YkR1HostTables { std::vector<int> lut; std::vector<uint16_t> rtab; std::vector<int16_t> r7; bool ok = false; };
static const YkR1HostTables& r1_host_tables() {
    static YkR1HostTables t;            // built once per process (thread-safe static initialisation), shared by every context
    static const bool built = [] {
        t.lut.assign((size_t)64 * YK_R1_R7MAX * YK_R1_LUT_INTS, 0);
        t.rtab.assign((size_t)64 * YK_R1_RTAB_R7 * 6 * YK_R1_RTAB_VALUES, 0);
        t.r7.assign((size_t)64 * YK_R1_R7_ROW, 0);
        for (int b6 = 0; b6 < 64; b6++) {
            const int BN = (b6 * YK_R1_BASE_MAX) / 63, scale = 223 - BN;
            for (int dd = 0; dd < YK_R1_R7_ROW; dd++) {                 // DiffRangeEncode with the clamped difference, EC.cpp:643-650 (C division)
                const int r7 = (dd * 127 + scale - 1) / scale;
                if (r7 < -32768 || r7 > 32767) return false;
                t.r7[(size_t)b6 * YK_R1_R7_ROW + dd] = (int16_t)r7;
            }
            for (int r7 = 0; r7 < YK_R1_R7MAX; r7++) {
                const int D = (r7 * scale) / 127 + 32;                 // DiffRangeDecode, EC.cpp:620-623
                const float DistNormF = (float)D;
                int* T = &t.lut[((size_t)b6 * YK_R1_R7MAX + r7) * YK_R1_LUT_INTS];
                for (int input = 0; input < 16; input++) {              // EC.cpp:662-677
                    float pos = input / 15.0f;
                    float ExpNormV = powf(pos, 1.4f), LogNormV = 1.0f - powf((1.0f - pos), 1.4f);
                    float outLinear = pos * DistNormF, outExp = ExpNormV * DistNormF, outLog = LogNormV * DistNormF;
                    T[input] = (int)(BN + outLinear); T[16 + input] = (int)(BN + outExp); T[32 + input] = (int)(BN + outLog);
                }
                for (int input = 0; input < 8; input++) {               // EC.cpp:680-696
                    float pos = input / 7.0f;
                    float ExpNormV = powf(pos, 1.4f), LogNormV = 1.0f - powf((1.0f - pos), 1.4f);
                    float outLinear = pos * DistNormF, outExp = ExpNormV * DistNormF, outLog = LogNormV * DistNormF;
                    T[48 + input] = (int)(BN + outLinear); T[56 + input] = (int)(BN + outExp); T[64 + input] = (int)(BN + outLog);
                }
                for (int m = 0; m < 6; m++) {
                    const int off = m < 3 ? 16 * m : 48 + 8 * (m - 3), count = m < 3 ? 16 : 8;
                    const int* L = T + off;
                    int* TH = T + 72 + off;
                    TH[0] = INT_MIN;
                    int next = INT_MAX;                                  // threshold of the next distinct entry
                    for (int n = count - 1; n >= 1; n--) {
                        if (L[n] < L[n - 1]) return false;                // never: every curve is monotone
                        if (r7 < YK_R1_RTAB_R7 && b6 < 63 && (L[n] > 255 || L[n - 1] < 0)) return false;     // never: BN + D <= 255 there
                        if (L[n] > L[n - 1]) next = (L[n - 1] + L[n]) >> 1;
                        TH[n] = next;
                    }
                    // the entry the search picks for every value of the tables' domain: code = #{n >= 1 : value > TH[n]}
                    if (r7 >= YK_R1_RTAB_R7 || b6 == 63) continue;      // range codes beyond 7 bits (a reference quirk for bases close to 224) and base 63 (entries up to 256) are searched
                    uint16_t* R = &t.rtab[(((size_t)b6 * YK_R1_RTAB_R7 + r7) * 6 + m) * YK_R1_RTAB_VALUES];
                    int code = 0;
                    for (int v = 0; v < YK_R1_RTAB_VALUES; v++) {
                        while (code + 1 < count && v > TH[code + 1]) code++;
                        R[v] = (uint16_t)((code << 8) | L[code]);
                    }
                }
            }
        }
        t.ok = true;
        return true;
    }();
    (void)built;
    return t;
}
static int ensure_r1_lut(yk_ctx* c) {
    if (c->lutDev && c->rtabDev && c->r7Dev) return YK_OK;
    if (c->noHostWait) return YK_ERR_STATE;
    const YkR1HostTables& t = r1_host_tables();
    if (!t.ok) return YK_ERR_STATE;
    CK(cudaMalloc((void**)&c->lutDev, t.lut.size() * sizeof(int)));
    CK(cudaMalloc((void**)&c->rtabDev, t.rtab.size() * sizeof(uint16_t)));
    CK(cudaMalloc((void**)&c->r7Dev, t.r7.size() * sizeof(int16_t)));
    // on the context's stream (non-blocking: it does not order itself after the legacy stream), complete before this returns
    cudaError_t e = cudaMemcpyAsync(c->lutDev, t.lut.data(), t.lut.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->rtabDev, t.rtab.data(), t.rtab.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->r7Dev, t.r7.data(), t.r7.size() * sizeof(int16_t), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
        cudaFree(c->lutDev); c->lutDev = nullptr; cudaFree(c->rtabDev); c->rtabDev = nullptr; cudaFree(c->r7Dev); c->r7Dev = nullptr;
        g_lastCuda = std::string("R1 table upload: ") + cudaGetErrorString(e); return YK_ERR_CUDA;
    }
    return YK_OK;
}

// DynamicTileEncode's walk over a plane of ph rows, halved on the axes of shX / shY, and its constraint box (cx, cy, cw, ch)
// to the caller.  The bound box is the alpha stage's once it has run (MipPrefilter), else the full image (CheckMipmapMask,
// EC.cpp:2784-2794).
static int r1_walk(yk_ctx* c, YkSlotHost& s, int ph, int shX, int shY, int constraint[4], YkR1Walk& g) {
    int rc;
    if (s.pendingHarvest) { rc = fetch_hdr(c, s); if (rc && rc != YK_ERR_RANGE) return rc; }
    int bound[4] = { 0, 0, s.d.w, s.d.h };
    if (s.alphaRan) { if ((rc = alpha_finish(c, s))) return rc; memcpy(bound, s.bound, sizeof bound); }
    g = yk_r1_walk(bound, ph, shX, shY);
    if (constraint) { constraint[0] = g.cx; constraint[1] = g.cy; constraint[2] = g.cw; constraint[3] = g.ch; }
    return YK_OK;
}

// one DynamicTileEncode launch pair (yk_k_r1_offsets + an encode kernel) on the context's stream
static int launch_r1(yk_ctx* c, int slot, const YkR1Launch& L) {
    YkSlotHost& s = c->slots[slot];
    int rc;
    if ((rc = ensure_r1_lut(c))) return rc;
    CK(cudaMemsetAsync(s.d.r1Status, 0, r1_status_words(s.d.w, s.d.h) * sizeof(unsigned long long), c->stream));
    { YkTimed t(c, 3); yk_launch_range_dyn_encode(c->slotsDev, slot, L, c->numSMs, c->lutDev, c->rtabDev, c->r7Dev, c->stream); }
    c->launches += 2;
    CK(cudaGetLastError());
    return YK_OK;
}

// the coded streams of plane `out` of the last DynamicTileEncode launch to the caller's buffers
static int r1_fetch(yk_ctx* c, YkSlotHost& s, int out, uint8_t* nibbles, int nibCap, int* nNibbles, uint16_t* defs, int defsCap, int* nDefs) {
    int tot[2] = { 0, 0 };
    CK(cudaMemcpyAsync(&tot[0], s.d.hdr + YK_HD_R1_NIB0 + out, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&tot[1], s.d.hdr + YK_HD_R1_DEF0 + out, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    const int nb = (tot[0] + 1) / 2;
    if (nNibbles) *nNibbles = tot[0];
    if (nDefs) *nDefs = tot[1];
    if (nb > nibCap || tot[1] > defsCap) return YK_ERR_CAPACITY;
    if (nibbles && nb) CK(cudaMemcpyAsync(nibbles, s.d.r1Nib[out], nb, cudaMemcpyDeviceToHost, c->stream));
    if (defs && tot[1]) CK(cudaMemcpyAsync(defs, s.d.r1Defs[out], (size_t)tot[1] * 2, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}

// DynamicTileEncode on one device plane (the slot's colour planes, or Y / reduced Co / Cg of the chroma front-end)
static int range_dyn_impl(yk_ctx* c, int slot, const int32_t* src, const uint8_t* srcU8, int pitchU8, int pw, int ph, int out, int mode3BitOnly, int chroma, int halfX, int halfY,
                          uint8_t* nibbles, int nibCap, int* nNibbles, uint16_t* defs, int defsCap, int* nDefs, int constraint[4], int32_t* dst) {
    YkSlotHost& s = c->slots[slot];
    const int w = s.d.w, h = s.d.h;
    if ((pw & 7) || (ph & 7)) return YK_ERR_ARG;
    YkR1Launch L;
    memset(&L, 0, sizeof L);
    L.nJobs = 1; L.mode3 = mode3BitOnly ? 1 : 0;
    L.pw = pw; L.ph = ph; L.shX = halfX ? 1 : 0; L.shY = halfY ? 1 : 0;
    int rc;
    if ((rc = r1_walk(c, s, ph, L.shX, L.shY, constraint, L.walk))) return rc;
    YkR1Args& a = L.job[0];
    a.src = src; a.srcU8 = srcU8; a.pitchU8 = pitchU8; a.chroma = chroma; a.out = out;
    // the optional full-size write-back plane: a device copy of the caller's plane, kept by the slot between calls
    if (dst) {
        if (!s.r1DstDev && (rc = dev_alloc(s, &s.r1DstDev, (size_t)c->maxW * c->maxH))) return rc;
        CK(cudaMemcpyAsync(s.r1DstDev, dst, (size_t)w * h * 4, cudaMemcpyHostToDevice, c->stream));
        a.dst = s.r1DstDev;
    }
    if ((rc = upload_slots(c, slot, 1))) return rc;
    s.r1Fused = 0;                                               // the streams of plane `out` are about to be replaced
    if ((rc = launch_r1(c, slot, L))) return rc;
    rc = r1_fetch(c, s, out, nibbles, nibCap, nNibbles, defs, defsCap, nDefs);
    if (!rc && dst) {
        CK(cudaMemcpyAsync(dst, s.r1DstDev, (size_t)w * h * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return rc;
}

// DynamicTileEncode of the three colour planes right behind the analysis, one launch, nothing comes back to the host:
// the constraint box is derived on the device from the alpha stage's box in the image header
static int enqueue_r1_fused(yk_ctx* c, int slot, int mode3BitOnly, bool useAlpha) {
    YkSlotHost& s = c->slots[slot];
    const int w = s.d.w, h = s.d.h;
    if ((w & 7) || (h & 7) || w < 32 || h < 32) return YK_ERR_ARG;      // the reference's own domain (SURVEY.md hazard 11)
    if (s.d.hasAbove || s.d.hasBelow) return YK_ERR_UNSUPPORTED;
    YkR1Launch L;
    memset(&L, 0, sizeof L);
    L.nJobs = 3; L.fromHdr = 1; L.useAlpha = useAlpha ? 1 : 0; L.mode3 = mode3BitOnly ? 1 : 0;
    L.pw = w; L.ph = h;
    const int full[4] = { 0, 0, w, h };
    L.walk = yk_r1_walk(full, h, 0, 0);                         // the largest possible box: the launch covers it
    for (int p = 0; p < 3; p++) {
        YkR1Args& a = L.job[p];
        a.src = s.d.plane[p]; a.srcU8 = s.d.isU8 ? s.d.planeU8[p] : nullptr; a.pitchU8 = s.d.pitchU8; a.out = p;
    }
    int rc;
    if ((rc = launch_r1(c, slot, L))) return rc;
    s.r1Fused = mode3BitOnly ? 2 : 1;
    return YK_OK;
}

extern "C" int yk_range_dyn(yk_ctx* c, int slot, int plane, int mode3BitOnly, uint8_t* nibbles, int nibCap, int* nNibbles,
                            uint16_t* defs, int defsCap, int* nDefs, int constraint[4], int32_t* dst) {
    if (!slot_ok(c, slot) || plane < 0 || plane > 2) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    int rc;
    if (s.strip) {
        // the strip's part of the image's streams, as the last yk_strip_range_dyn / yk_strip_run_stages coded them
        if (dst) return YK_ERR_UNSUPPORTED;
        if (s.r1Strip != (mode3BitOnly ? 2 : 1)) return YK_ERR_STATE;
        if (constraint) memcpy(constraint, s.r1StripConstraint, sizeof s.r1StripConstraint);
        return r1_fetch(c, s, plane, nibbles, nibCap, nNibbles, defs, defsCap, nDefs);
    }
    if (!dst && s.r1Fused == (mode3BitOnly ? 2 : 1)) {
        // coded by yk_analyze already: only the streams come back
        YkR1Walk g;
        if ((rc = r1_walk(c, s, s.d.h, 0, 0, constraint, g))) return rc;
        return r1_fetch(c, s, plane, nibbles, nibCap, nNibbles, defs, defsCap, nDefs);
    }
    // samples outside 0..255 were uploaded as int32 by yk_set_image; packed planes are read as bytes
    const bool u8 = s.d.isU8 != 0;
    if (!u8 && !s.int32Valid && (rc = ensure_int32(c, slot))) return rc;
    return range_dyn_impl(c, slot, s.d.plane[plane], u8 ? s.d.planeU8[plane] : nullptr, s.d.pitchU8, s.d.w, s.d.h, plane, mode3BitOnly, 0, 0, 0,
                          nibbles, nibCap, nNibbles, defs, defsCap, nDefs, constraint, dst);
}

// ---- chroma front-end (SURVEY.md 8f row 3) ----------------------------------------------------------------
extern "C" int yk_chroma_prepare(yk_ctx* c, int slot, const int half[4], const int downMode[2]) {
    if (!slot_ok(c, slot) || !half || !downMode) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    const int w = s.d.w, h = s.d.h;
    if ((w & 1) || (h & 1)) return YK_ERR_ARG;
    for (int k = 0; k < 2; k++) {
        const int hx = half[2 * k] != 0, hy = half[2 * k + 1] != 0, m = downMode[k];
        if (m < 0 || m > 4) return YK_ERR_ARG;
        // NEAREST_BR / MAX_BOX / MIN_BOX on one axis read the sample past the plane in the reference (Plane.cpp:297-356)
        if ((hx != hy) && (m == 1 || m == 3 || m == 4)) return YK_ERR_UNSUPPORTED;
    }
    CK(cudaSetDevice(c->device));
    int rc;
    if ((rc = ensure_int32(c, slot))) return rc;
    for (int k = 0; k < 3; k++)
        if (!s.chroma[k]) { if ((rc = dev_alloc(s, &s.chroma[k], (size_t)c->maxW * c->maxH))) return rc; }
    YkChromaArgs a;
    a.y = s.chroma[0]; a.co = s.chroma[1]; a.cg = s.chroma[2];
    for (int k = 0; k < 4; k++) { a.half[k] = half[k] != 0; s.chromaHalf[k] = a.half[k]; }
    a.mode[0] = downMode[0]; a.mode[1] = downMode[1];
    if ((rc = upload_slots(c, slot, 1))) return rc;
    { YkTimed t(c, 4); yk_launch_chroma(c->slotsDev, slot, w, h, a, c->stream); }
    c->launches += 1;
    CK(cudaGetLastError());
    s.chromaReady = true;
    return YK_OK;
}

static void chroma_dims(const YkSlotHost& s, int which, int* pw, int* ph) {
    const int hx = which ? s.chromaHalf[2 * (which - 1)] : 0, hy = which ? s.chromaHalf[2 * (which - 1) + 1] : 0;
    *pw = hx ? s.d.w / 2 : s.d.w; *ph = hy ? s.d.h / 2 : s.d.h;
}

extern "C" int yk_chroma_plane(yk_ctx* c, int slot, int which, int32_t* out, int* outW, int* outH) {
    if (!slot_ok(c, slot) || which < 0 || which > 2) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.chromaReady) return YK_ERR_STATE;
    int pw, ph;
    chroma_dims(s, which, &pw, &ph);
    if (outW) *outW = pw;
    if (outH) *outH = ph;
    if (out) {
        CK(cudaSetDevice(c->device));
        CK(cudaMemcpyAsync(out, s.chroma[which], (size_t)pw * ph * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return YK_OK;
}

extern "C" int yk_range_dyn_chroma(yk_ctx* c, int slot, int which, int mode3BitOnly, uint8_t* nibbles, int nibCap, int* nNibbles,
                                   uint16_t* defs, int defsCap, int* nDefs, int constraint[4], int32_t* dst) {
    if (!slot_ok(c, slot) || which < 0 || which > 2) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.chromaReady) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    int pw, ph;
    chroma_dims(s, which, &pw, &ph);
    const int hx = pw != s.d.w, hy = ph != s.d.h;
    return range_dyn_impl(c, slot, s.chroma[which], nullptr, 0, pw, ph, which, mode3BitOnly, which != 0, hx, hy, nibbles, nibCap, nNibbles, defs, defsCap, nDefs, constraint, dst);
}

// ---- compat state download --------------------------------------------------------------------------------
extern "C" int yk_download_state(yk_ctx* c, int slot, int32_t* smoothMap, int32_t* const* mapSmoothTile,
                                 int32_t* const* mappedRGB, int32_t* mipmapMask, int32_t* const* recon) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    if (s.alphaRan && !s.alphaFetched) { int rc = alpha_finish(c, s); if (rc) return rc; }
    int rc = upload_slots(c, slot, 1);
    if (rc) return rc;
    if (recon && (rc = ensure_int32(c, slot))) return rc;
    const size_t n = (size_t)s.d.w * s.d.h, n1 = (size_t)(s.d.w + 1) * (s.d.h + 1);
    struct Tmp { int32_t* p = nullptr; ~Tmp() { if (p) cudaFree(p); } } gSmooth, gMask, gMapped, gRec;     // freed on every way out
    int32_t *&dSmooth = gSmooth.p, *&dMask = gMask.p, *&dMapped = gMapped.p, *&dRec = gRec.p;
    const bool wantSmooth = smoothMap || mapSmoothTile, wantRec = recon != nullptr;
    if (wantSmooth) CK(cudaMalloc((void**)&dSmooth, n * 4));
    if (mipmapMask) CK(cudaMalloc((void**)&dMask, n * 4));
    if (mappedRGB) CK(cudaMalloc((void**)&dMapped, n1 * 4));
    if (wantRec) CK(cudaMalloc((void**)&dRec, 3 * n * 4));
    yk_launch_state(c->slotsDev, slot, s.d.nbx * s.d.nby, dSmooth, dMask, dMapped, dRec, dRec ? dRec + n : nullptr, dRec ? dRec + 2 * n : nullptr, c->stream);
    c->launches++;
    CK(cudaGetLastError());
    if (smoothMap) CK(cudaMemcpyAsync(smoothMap, dSmooth, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (mapSmoothTile) for (int p = 0; p < 3; p++) if (mapSmoothTile[p]) CK(cudaMemcpyAsync(mapSmoothTile[p], dSmooth, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (mipmapMask) CK(cudaMemcpyAsync(mipmapMask, dMask, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (mappedRGB) for (int p = 0; p < 3; p++) if (mappedRGB[p]) CK(cudaMemcpyAsync(mappedRGB[p], dMapped, n1 * 4, cudaMemcpyDeviceToHost, c->stream));
    if (recon) for (int p = 0; p < 3; p++) if (recon[p]) CK(cudaMemcpyAsync(recon[p], dRec + p * n, n * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}

extern "C" int yk_result_bytes(yk_ctx* c, int slot, long long out[6]) {
    if (!slot_ok(c, slot) || !out) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    int rc = fetch_hdr(c, s);
    if (rc) return rc;
    const int w = s.d.w, h = s.d.h;
    long long bm = 0, rgb = 0;
    for (int p = 0; p < YK_NPASS; p++) {
        const YkPassGeom& g = kGeom[p];
        bm += (long long)((w + g.bw - 1) / g.bw) * ((h + g.bh - 1) / g.bh) * g.bits / 8;
        rgb += s.hdr[YK_HD_PASS0 + p * YK_ST_STRIDE + YK_ST_RGBBYTES];
    }
    out[0] = bm; out[1] = rgb;
    out[2] = 3ll * 16 * s.hdr[YK_HD_R2_CHUNKS]; out[3] = 3ll * 3 * s.hdr[YK_HD_R2_TILES];
    out[4] = s.d.nPlanes == 4 ? ((long long)((w + 15) / 16) * ((h + 15) / 16) + 7) / 8 : 0;
    out[5] = 0;
    return YK_OK;
}

// ---- everything at once, without further copies -----------------------------------------------------------
extern "C" int yk_fetch_all(yk_ctx* c, int slot, yk_results* out) {
    if (!slot_ok(c, slot) || !out) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.k1Ran) return YK_ERR_STATE;
    int rc = harvest(c, s);
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    const int w = s.d.w;
    for (int p = 0; p < YK_NPASS; p++) {
        if (!(s.arMask & (1 << p))) continue;
        const int* st = s.hdr + YK_HD_PASS0 + p * YK_ST_STRIDE;
        out->bitmap[p] = s.arena + s.arBitmap[p]; out->bitmapBytes[p] = (int)pass_bitmap_bytes(s, p);
        out->rgb[p] = s.arena + s.arRgb[p]; out->rgbBytes[p] = st[YK_ST_RGBBYTES];
        out->tileDone[p] = st[YK_ST_TILEDONE];
        out->bbox[p][0] = w - st[YK_ST_MINX]; out->bbox[p][1] = st[YK_ST_MINY] ? INT_MAX / 2 - st[YK_ST_MINY] : s.d.imgH;
        out->bbox[p][2] = st[YK_ST_MAXX]; out->bbox[p][3] = st[YK_ST_MAXY];
    }
    if (s.arR2) {
        out->r2IdxBytes = 16 * s.hdr[YK_HD_R2_CHUNKS]; out->r2TypeBytes = 3 * s.hdr[YK_HD_R2_TILES];
        for (int pl = 0; pl < 3; pl++) { out->r2Idx[pl] = s.arena + s.arIdx[pl]; out->r2Type[pl] = s.arena + s.arType[pl]; }
    }
    if (s.alphaRan && s.d.nPlanes == 4 && !s.d.hasAbove && !s.d.hasBelow) {
        rc = alpha_finish(c, s);
        if (rc == YK_OK) {
            out->alphaValid = 1;
            out->alphaBitmap = s.alphaBitmap.empty() ? nullptr : s.alphaBitmap.data(); out->alphaBitmapBytes = (int)s.alphaBitmap.size();
            memcpy(out->alphaBound, s.bound, sizeof s.bound); memcpy(out->alphaChunkBBox, s.chunkBBox, sizeof s.chunkBBox);
            out->alphaRemaining = s.remaining; out->alphaWroteChunk = s.wroteChunk;
        }
    }
    return YK_OK;
}

// ---- multi-GPU: tile-row strips of one large image (SURVEY.md 8e) ----------------------------------------
extern "C" int yk_strip_config(yk_ctx* c, int slot, int imgH, int y0) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage) return YK_ERR_STATE;
    const int w = s.d.w, h = s.d.h;
    if (imgH < h || y0 < 0 || y0 + h > imgH || (y0 & 63)) return YK_ERR_ARG;
    if (y0 + h < imgH && (h & 63)) return YK_ERR_ARG;            // only the last strip may end off the 64-row grid
    CK(cudaSetDevice(c->device));
    const size_t es = s.d.isU8 ? 1 : sizeof(int32_t), rowBytes = ((size_t)w * es + 15) / 16 * 16;
    const size_t touchBytes = ((size_t)s.d.latW * sizeof(uint32_t) + 15) / 16 * 16;
    const size_t need = 3 * rowBytes + 2 * touchBytes + 64;
    if (s.haloBytes < need) {
        if (s.haloIn) cudaFree(s.haloIn);
        s.haloIn = nullptr; s.haloBytes = 0;
        CK(cudaMalloc((void**)&s.haloIn, need));
        s.haloBytes = need;
    }
    // complete before this returns: the neighbour strips write into this buffer from other streams / processes, and
    // nothing else orders their copies after a clear still queued here
    CK(cudaMemsetAsync(s.haloIn, 0, need, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    s.d.imgH = imgH; s.d.y0 = y0;
    s.d.hasAbove = y0 > 0; s.d.hasBelow = y0 + h < imgH;
    for (int p = 0; p < 3; p++) s.d.rowBelow[p] = s.d.hasBelow ? (const void*)(s.haloIn + p * rowBytes) : nullptr;
    s.d.touchInTop = (const uint32_t*)(s.haloIn + 3 * rowBytes);
    s.d.touchInBottom = (const uint32_t*)(s.haloIn + 3 * rowBytes + touchBytes);
    s.haloFlagsOffset = 3 * rowBytes + 2 * touchBytes;
    s.stripEpoch = 0; s.peerAbove = nullptr; s.peerBelow = nullptr;
    s.strip = true; s.r1Strip = 0;
    s.dirty = true;
    return YK_OK;
}

extern "C" int yk_strip_halo_ptrs(yk_ctx* c, int slot, yk_strip_halo* out) {
    if (!slot_ok(c, slot) || !out) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.haloIn) return YK_ERR_STATE;
    const int w = s.d.w;
    memset(out, 0, sizeof *out);
    out->haloIn = s.haloIn; out->haloBytes = s.haloBytes;
    const size_t es = s.d.isU8 ? 1 : sizeof(int32_t), rowBytes = ((size_t)w * es + 15) / 16 * 16;
    out->pixelRowInOffset = 0; out->pixelRowBytes = 3 * rowBytes; out->pixelRowStride = rowBytes;
    out->touchInTopOffset = out->pixelRowBytes;
    out->touchBytes = (size_t)s.d.latW * sizeof(uint32_t);
    out->touchInBottomOffset = (size_t)((const uint8_t*)s.d.touchInBottom - s.haloIn);
    for (int p = 0; p < 3; p++) out->pixelRowOut[p] = s.d.isU8 ? (const void*)s.d.planeU8[p] : (const void*)s.d.plane[p];   // first pixel row of each colour plane
    out->planeRowBytes = (size_t)w * es;
    out->touchOutTop = s.d.touchMap;                                                         // lattice row 0
    out->touchOutBottom = s.d.touchMap + (size_t)(s.d.latH - 1) * s.d.latW;                  // lattice row h/4
    return YK_OK;
}

extern "C" int yk_strip_phase(yk_ctx* c, int slot, int phase, int rejectFactor) {
    if (!slot_ok(c, slot) || (phase != 0 && phase != 1) || rejectFactor < 0 || rejectFactor > 64) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.haloIn) return YK_ERR_STATE;
    YkRun run; memset(&run, 0, sizeof run);
    run.rejectFactor = rejectFactor;
    run.doAlpha = s.d.nPlanes == 4;
    run.nPasses = YK_NPASS; for (int i = 0; i < YK_NPASS; i++) run.passId[i] = i;
    if (phase == 0) {
        if (s.prepared || s.nextPass || !s.cellsClean) return YK_ERR_STATE;         // needs a fresh state
        return enqueue(c, slot, 1, run, true, true, 1);
    }
    if (s.cellsClean || s.prepared) return YK_ERR_STATE;                            // phase 0 first, once
    const int rc = enqueue(c, slot, 1, run, true, true, 2);
    if (rc) return rc;
    s.prepared = true; s.preparedReject = rejectFactor; s.nextPass = 0;
    return YK_OK;
}

// ---- DynamicTileEncode of a strip -----------------------------------------------------------------------------------
// An 8x8 block depends on its own samples, its 4x4 cells' claimed bits (final after phase 0) and the alpha mask, and strips
// start on multiples of 64: each strip codes the blocks of the image's walk whose top row it holds, with the image's
// geometry.  The image's constraint box and the mask decision are the only global inputs (imageBoundPx: the strip set's
// merged alpha box, or the whole image).  Each strip's streams start at 0; concatenated in strip order they are the image's.
static int r1_strip_args(const YkSlotHost& s, const int imageBoundPx[4]) {
    const int w = s.d.w, imgH = s.d.imgH;
    if ((w & 7) || (imgH & 7) || w < 32 || imgH < 32) return YK_ERR_ARG;      // the reference's own domain (SURVEY.md hazard 11)
    if ((s.d.nPlanes == 4) != (imageBoundPx != nullptr)) return YK_ERR_ARG;   // RGBA: the merged alpha box; RGB: the whole image
    if (imageBoundPx) {
        const int L = imageBoundPx[0], T = imageBoundPx[1], R = imageBoundPx[2], B = imageBoundPx[3];
        if (L < 0 || T < 0 || R > w || B > imgH || L >= R || T >= B) return YK_ERR_ARG;
    }
    return YK_OK;
}

// enqueues the three-plane pair (yk_k_r1_offsets + yk_k_r1_encode3) over the strip's window; no synchronisation
static int enqueue_r1_strip(yk_ctx* c, int slot, int mode3BitOnly, const int imageBoundPx[4]) {
    YkSlotHost& s = c->slots[slot];
    const int w = s.d.w, imgH = s.d.imgH;
    const int full[4] = { 0, 0, w, imgH };
    const int* box = imageBoundPx ? imageBoundPx : full;
    // mipmapMask holds the alpha stage's rejection unless the box is the whole image (EC.cpp:1400-1403)
    const int maskValid = s.d.nPlanes == 4, maskReset = maskValid && yk_box_is_image(box, w, imgH);
    if (s.d.alphaValid != maskValid || s.d.alphaReset != maskReset) { s.d.alphaValid = maskValid; s.d.alphaReset = maskReset; s.dirty = true; }
    int rc;
    if ((rc = upload_slots(c, slot, 1))) return rc;
    YkR1Launch L;
    memset(&L, 0, sizeof L);
    L.nJobs = 3; L.mode3 = mode3BitOnly ? 1 : 0;
    L.pw = w; L.ph = imgH;
    const YkR1Walk g = yk_r1_walk(box, imgH, 0, 0);
    L.walk = yk_r1_window(g, s.d.y0, s.d.h);
    for (int p = 0; p < 3; p++) {
        YkR1Args& a = L.job[p];
        a.src = s.d.plane[p]; a.srcU8 = s.d.isU8 ? s.d.planeU8[p] : nullptr; a.pitchU8 = s.d.pitchU8; a.out = p;
    }
    s.r1Strip = 0;                                               // the streams are about to be replaced
    if ((rc = launch_r1(c, slot, L))) return rc;
    s.r1Strip = mode3BitOnly ? 2 : 1;
    s.r1StripConstraint[0] = g.cx; s.r1StripConstraint[1] = g.cy; s.r1StripConstraint[2] = g.cw; s.r1StripConstraint[3] = g.ch;
    return YK_OK;
}

extern "C" int yk_strip_range_dyn(yk_ctx* c, int slot, int mode3BitOnly, const int imageBoundPx[4]) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.strip) return YK_ERR_STATE;
    int rc;
    if ((rc = r1_strip_args(s, imageBoundPx))) return rc;
    if (s.cellsClean) return YK_ERR_STATE;                         // phase 0 has not run on this image
    CK(cudaSetDevice(c->device));
    return enqueue_r1_strip(c, slot, mode3BitOnly, imageBoundPx);
}

// ---- strips without the host in the loop ----------------------------------------------------------------------------
// Every strip enqueues the whole image on its own stream: the two exchanges are device-to-device copies into the
// neighbours' halo allocations (peer-mapped: NVLink P2P), each followed by a one-thread kernel that publishes an epoch
// number in the neighbour's halo; before it uses what a neighbour sends, a strip's stream runs a one-thread kernel that
// waits for that number.  No host barrier, no collective.  Flags (u32, in the strip's own halo, written by neighbours):
//   [0] pixel row of the strip below has landed        [1] touch words of the strip above   [2] touch words of the strip below
//   [3] the strip above has finished the image         [4] the strip below has finished the image
extern "C" int yk_strip_set_peers(yk_ctx* c, int slot, void* aboveHalo, void* belowHalo) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.haloIn) return YK_ERR_STATE;
    if ((s.d.hasAbove && !aboveHalo) || (s.d.hasBelow && !belowHalo)) return YK_ERR_ARG;
    // the R1 tables go up now, while waiting for this stream is harmless: yk_strip_run_stages must not wait
    CK(cudaSetDevice(c->device));
    const int rc = ensure_r1_lut(c);
    if (rc) return rc;
    s.peerAbove = s.d.hasAbove ? aboveHalo : nullptr; s.peerBelow = s.d.hasBelow ? belowHalo : nullptr;
    return YK_OK;
}

static int strip_run_check(yk_ctx* c, int slot, int rejectFactor, int stages) {
    if (!slot_ok(c, slot) || rejectFactor < 0 || rejectFactor > 64) return YK_ERR_ARG;
    const int r1 = stages & (YK_STAGE_RANGEDYN | YK_STAGE_RANGEDYN3);
    if ((stages & ~r1) || r1 == (YK_STAGE_RANGEDYN | YK_STAGE_RANGEDYN3)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.haloIn) return YK_ERR_STATE;
    if ((s.d.hasAbove && !s.peerAbove) || (s.d.hasBelow && !s.peerBelow)) return YK_ERR_STATE;
    // RGBA: the alpha box is a reduction over every strip, not a neighbour exchange
    if (r1 && s.d.nPlanes == 4) return YK_ERR_UNSUPPORTED;
    if (r1) return r1_strip_args(s, nullptr);
    return YK_OK;
}

struct YkNoHostWait {       // see yk_ctx::noHostWait
    yk_ctx* c;
    explicit YkNoHostWait(yk_ctx* c_) : c(c_) { c->noHostWait = true; }
    ~YkNoHostWait() { c->noHostWait = false; }
};

static int strip_run_enqueue(yk_ctx* c, int slot, int rejectFactor, int stages) {
    YkSlotHost& s = c->slots[slot];
    CK(cudaSetDevice(c->device));
    // Nothing below may make the host wait for this stream: it is about to hold kernels that wait for the neighbours,
    // whose work the same host thread may still have to enqueue.  So the slot descriptor goes up now (a copy from
    // pageable memory drains the stream first), with the mask flags yk_reset_state below clears, and the previous
    // image's header is not fetched (its counters are lost unless they were read before the next run).
    if (s.d.alphaValid || s.d.alphaReset) { s.d.alphaValid = 0; s.d.alphaReset = 0; s.dirty = true; }
    int rc = upload_slots(c, slot, 1);
    if (rc) return rc;
    s.pendingHarvest = false;
    YkNoHostWait guard(c);
    const unsigned e = ++s.stripEpoch;
    const size_t es = s.d.isU8 ? 1 : sizeof(int32_t), rowBytes = ((size_t)s.d.w * es + 15) / 16 * 16;
    const size_t touchBytes = (size_t)s.d.latW * sizeof(uint32_t);
    const size_t offTop = (size_t)((const uint8_t*)s.d.touchInTop - s.haloIn), offBottom = (size_t)((const uint8_t*)s.d.touchInBottom - s.haloIn);
    unsigned* mine = (unsigned*)(s.haloIn + s.haloFlagsOffset);
    unsigned* above = s.peerAbove ? (unsigned*)((uint8_t*)s.peerAbove + s.haloFlagsOffset) : nullptr;     // same layout: same width and sample type
    unsigned* below = s.peerBelow ? (unsigned*)((uint8_t*)s.peerBelow + s.haloFlagsOffset) : nullptr;
    // the neighbours have finished the previous image: their halos may be overwritten, and they have read what we sent
    if (e > 1 && (above || below)) { yk_launch_flag_wait(above ? mine + 3 : nullptr, below ? mine + 4 : nullptr, e - 1, c->stream); c->launches++; }
    if ((rc = yk_reset_state(c, slot))) return rc;
    // exchange 1: my first pixel row -> halo of the strip above
    if (above) {
        for (int p = 0; p < 3; p++) {
            const void* src = s.d.isU8 ? (const void*)s.d.planeU8[p] : (const void*)s.d.plane[p];
            CK(cudaMemcpyAsync((uint8_t*)s.peerAbove + p * rowBytes, src, (size_t)s.d.w * es, cudaMemcpyDefault, c->stream));
        }
        yk_launch_flag_set(above + 0, nullptr, e, c->stream); c->launches++;
    }
    if (below) { yk_launch_flag_wait(mine + 0, nullptr, e, c->stream); c->launches++; }
    if ((rc = yk_strip_phase(c, slot, 0, rejectFactor))) return rc;
    // exchange 2: boundary touch words, both directions
    if (above) CK(cudaMemcpyAsync((uint8_t*)s.peerAbove + offBottom, s.d.touchMap, touchBytes, cudaMemcpyDefault, c->stream));
    if (below) CK(cudaMemcpyAsync((uint8_t*)s.peerBelow + offTop, s.d.touchMap + (size_t)(s.d.latH - 1) * s.d.latW, touchBytes, cudaMemcpyDefault, c->stream));
    if (above || below) { yk_launch_flag_set(above ? above + 2 : nullptr, below ? below + 1 : nullptr, e, c->stream); c->launches++; }
    // R1 needs nothing from the neighbours: it runs while their touch words travel
    if ((stages & (YK_STAGE_RANGEDYN | YK_STAGE_RANGEDYN3)) && (rc = enqueue_r1_strip(c, slot, (stages & YK_STAGE_RANGEDYN3) != 0, nullptr))) return rc;
    if (above || below) { yk_launch_flag_wait(above ? mine + 1 : nullptr, below ? mine + 2 : nullptr, e, c->stream); c->launches++; }
    if ((rc = yk_strip_phase(c, slot, 1, rejectFactor))) return rc;
    if (above || below) { yk_launch_flag_set(above ? above + 4 : nullptr, below ? below + 3 : nullptr, e, c->stream); c->launches++; }
    CK(cudaGetLastError());
    return YK_OK;
}

extern "C" int yk_strip_run_stages(yk_ctx* c, int slot, int rejectFactor, int stages) {
    const int rc = strip_run_check(c, slot, rejectFactor, stages);
    if (rc) return rc;
#ifdef YK_EMULATE
    return YK_ERR_UNSUPPORTED;      // the emulated launches run to completion one after the other: a waiting kernel would never see its flag
#endif
    return strip_run_enqueue(c, slot, rejectFactor, stages);
}
extern "C" int yk_strip_run(yk_ctx* c, int slot, int rejectFactor) { return yk_strip_run_stages(c, slot, rejectFactor, 0); }

// all strips of an image driven by this process (one context per strip, on one or several GPUs): link every strip to its
// neighbours' halo allocations directly, then enqueue an image on every strip
extern "C" int yk_strips_link(yk_ctx* const* ctxs, int n, int slot) {
    if (!ctxs || n < 1) return YK_ERR_ARG;
    for (int k = 0; k < n; k++) if (!slot_ok(ctxs[k], slot) || !ctxs[k]->slots[slot].haloIn) return YK_ERR_STATE;
#ifndef YK_EMULATE
    for (int k = 0; k + 1 < n; k++) {
        const int a = ctxs[k]->device, b = ctxs[k + 1]->device;
        if (a == b) continue;
        int ok1 = 0, ok2 = 0;
        CK(cudaDeviceCanAccessPeer(&ok1, a, b)); CK(cudaDeviceCanAccessPeer(&ok2, b, a));
        if (!ok1 || !ok2) return YK_ERR_UNSUPPORTED;
        cudaError_t e;
        CK(cudaSetDevice(a)); e = cudaDeviceEnablePeerAccess(b, 0); if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e); cudaGetLastError();
        CK(cudaSetDevice(b)); e = cudaDeviceEnablePeerAccess(a, 0); if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e); cudaGetLastError();
    }
#endif
    for (int k = 0; k < n; k++) {
        const int rc = yk_strip_set_peers(ctxs[k], slot, k > 0 ? ctxs[k - 1]->slots[slot].haloIn : nullptr, k + 1 < n ? ctxs[k + 1]->slots[slot].haloIn : nullptr);
        if (rc) return rc;
    }
    return YK_OK;
}
extern "C" int yk_strips_run_stages(yk_ctx* const* ctxs, int n, int slot, int rejectFactor, int stages) {
    if (!ctxs || n < 1) return YK_ERR_ARG;
    for (int k = 0; k < n; k++) { const int rc = strip_run_check(ctxs[k], slot, rejectFactor, stages); if (rc) return rc; }     // nothing enqueued on an error
    for (int k = 0; k < n; k++) { const int rc = yk_strip_run_stages(ctxs[k], slot, rejectFactor, stages); if (rc) return rc; }
    return YK_OK;
}
extern "C" int yk_strips_run(yk_ctx* const* ctxs, int n, int slot, int rejectFactor) { return yk_strips_run_stages(ctxs, n, slot, rejectFactor, 0); }

// ---- alpha stage of a strip set: the per-tile results of one strip, and their assembly (host code) ------------------
extern "C" int yk_alpha_kept(yk_ctx* c, int slot, uint8_t* kept, int keptCap, int* tilesW, int* tilesH, int boundPx[4], int* keptTiles) {
    if (!slot_ok(c, slot)) return YK_ERR_ARG;
    YkSlotHost& s = c->slots[slot];
    if (!s.haveImage || !s.alphaRan || s.d.nPlanes != 4) return YK_ERR_STATE;
    CK(cudaSetDevice(c->device));
    int rc = fetch_hdr(c, s);
    if (rc) return rc;
    const int tw = (s.d.w + 15) / 16, th = (s.d.h + 15) / 16;
    if (tilesW) *tilesW = tw;
    if (tilesH) *tilesH = th;
    if (keptTiles) *keptTiles = s.hdr[YK_HD_ALPHA_KEPT0];
    if (boundPx) yk_alpha_box(s.hdr, s.d.w, boundPx);
    if (kept) {
        if (keptCap < tw * th) return YK_ERR_CAPACITY;
        CK(cudaMemcpyAsync(kept, s.d.alphaKept, (size_t)tw * th, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return YK_OK;
}

// MipPrefilter's results (EC.cpp:1287-1403) from the per-tile "kept" bytes of a whole image ([tilesH][tilesW], e.g. the
// strips' arrays one after the other) and the bound box of the kept tiles: bitmap over the box, remaining pixels, chunk box
extern "C" int yk_alpha_assemble(const uint8_t* kept, int tilesW, int tilesH, int w, int h, const int boundPx[4],
                                 uint8_t* bitmap, int bitmapCap, int* bitmapBytes, int* remainingPixels, int* wroteChunk, int chunkBBoxTiles[4]) {
    if (!kept || !boundPx || tilesW < 1 || tilesH < 1 || !bitmapBytes) return YK_ERR_ARG;
    const int L = boundPx[0], T = boundPx[1], R = boundPx[2], B = boundPx[3];
    *bitmapBytes = 0;
    if (L == 0 && T == 0 && R == w && B == h) {                    // EC.cpp:1400-1403: the rejection is discarded
        if (remainingPixels) *remainingPixels = R * B;
        if (wroteChunk) *wroteChunk = 0;
        return YK_OK;
    }
    const int bx0 = L >> 4, bx1 = (R + 15) >> 4, by0 = T >> 4, by1 = (B + 15) >> 4;
    const int tWB = bx1 - bx0, tHB = by1 - by0, nb = (tWB * tHB + 7) / 8;
    if (tWB <= 0 || tHB <= 0 || bx1 > tilesW || by1 > tilesH) return YK_ERR_ARG;
    if (nb > bitmapCap || !bitmap) return YK_ERR_CAPACITY;
    memset(bitmap, 0, (size_t)nb);
    int bit = 0, rem = 0;
    for (int y = 0; y < tHB; y++)
        for (int x = 0; x < tWB; x++, bit++)
            if (kept[(size_t)(y + by0) * tilesW + x + bx0]) { bitmap[bit >> 3] |= (uint8_t)(1 << (bit & 7)); rem += 256; }   // EC.cpp:1317-1327
    *bitmapBytes = nb;
    if (remainingPixels) *remainingPixels = rem;
    if (wroteChunk) *wroteChunk = 1;
    if (chunkBBoxTiles) { chunkBBoxTiles[0] = bx0; chunkBBoxTiles[1] = by0; chunkBBoxTiles[2] = tWB; chunkBBoxTiles[3] = tHB; }
    return YK_OK;
}

// ---- peer-to-peer plumbing for the halo exchange: CUDA IPC handles of the halo buffers and plain async copies
// (device to device, peer access over NVLink when the two GPUs allow it; no collective)
extern "C" int yk_ipc_export(const void* devPtr, unsigned char handle[64]) {
    if (!devPtr || !handle) return YK_ERR_ARG;
#ifdef YK_EMULATE
    memset(handle, 0, 64); memcpy(handle, &devPtr, sizeof devPtr);
    return YK_OK;
#else
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, (void*)devPtr));
    memcpy(handle, &h, 64);
    return YK_OK;
#endif
}
extern "C" int yk_ipc_open(yk_ctx* c, const unsigned char handle[64], void** devPtr) {
    if (!c || !handle || !devPtr) return YK_ERR_ARG;
#ifdef YK_EMULATE
    memcpy(devPtr, handle, sizeof *devPtr);
    return YK_OK;
#else
    CK(cudaSetDevice(c->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CK(cudaIpcOpenMemHandle(devPtr, h, cudaIpcMemLazyEnablePeerAccess));
    return YK_OK;
#endif
}
extern "C" int yk_ipc_close(yk_ctx* c, void* devPtr) {
    if (!c || !devPtr) return YK_ERR_ARG;
#ifndef YK_EMULATE
    CK(cudaSetDevice(c->device));
    CK(cudaIpcCloseMemHandle(devPtr));
#endif
    return YK_OK;
}
extern "C" int yk_copy_async(yk_ctx* c, void* dst, const void* src, size_t bytes) {
    if (!c || !dst || !src) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, c->stream));
    return YK_OK;
}
// host <-> device copies of halo data for transports that stage through the host (and for tests)
extern "C" int yk_copy_to_host(yk_ctx* c, void* hostDst, const void* devSrc, size_t bytes) {
    if (!c || !hostDst || !devSrc) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(hostDst, devSrc, bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}
extern "C" int yk_copy_from_host(yk_ctx* c, void* devDst, const void* hostSrc, size_t bytes) {
    if (!c || !devDst || !hostSrc) return YK_ERR_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpyAsync(devDst, hostSrc, bytes, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return YK_OK;
}
