// yaik_b200 — yk_k_analyze: the persistent, TMA-staged analysis kernel (sm_100a).
//
// What the reference computes sequentially, tile after tile in stream order (KLab/YAIK, encoder/EncoderContext.cpp =
// "EC.cpp"), is restated in order-free form so that a 64x64 region (the largest swizzle block,
// include/YAIK_private.h:212-276) can be analysed independently of every other region:
//
//   MipPrefilter/quadRecursion (EC.cpp:1257-1427, 357-430)   per 16x16 tile "all alpha == 0", by ballot
//   FittingQuadSmooth accept decisions (EC.cpp:3810-3998)    all 7 passes of the region; tiles of every shape nest in an
//                                                            aligned 16x16 macro tile and eligibility only looks at the
//                                                            tile's own top-left cell, so one warp runs the whole cascade
//                                                            of a macro tile without any block barrier
//   DynamicTileCompressor (EC.cpp:8398-8522)                 the four 8x8 tiles of the macro tile are coded by the same warp
//                                                            right after its cascade (their cells are final by then), from
//                                                            the pixels already in shared memory, into a fixed per-tile
//                                                            place; yk_k_emit moves them to their stream offsets
//
// Structure: one CTA per SM, persistent.  The unit of work is one macro-tile row of two neighbouring regions (128 x 16
// pixels, eight macro tiles; the TMA unit's service time is per box row, about 22 cycles for rows up to 528 bytes, so the
// boxes are made wide), taken by global ticket.  One producer warp takes tickets — never more than a few units ahead of the consumers,
// so the CTAs finish together — and issues the TMA box loads (cp.async.bulk.tensor, one per plane: 17 x 132 int32 samples
// per colour plane, 16 x 128 alpha) into a ring of raw staging buffers, completion on an mbarrier per buffer.
// 23 consumer warps take macro tiles from a block-local queue: a warp packs its macro tile's 17x17x3 samples to bytes
// into a warp-private tile (clamped the way Plane::GetPixelValue clamps), tests its alpha tile, releases the raw buffer,
// then runs the cascade and the range stage out of the private tile and writes the macro tile's results straight to
// global memory (accept bits, claimed cells and touch words by atomic OR).  Per-pass counters are summed per CTA.
// No block-wide barrier after start-up; every wait is an mbarrier try_wait (the hardware suspends the warp).
//
// No tensor cores: the work is integer min/max reductions over bytes, bounded by HBM and the integer pipes.
#include "yk_device.h"

#ifndef YKA_NR
#define YKA_NR 4                    // raw staging buffers (TMA destinations), one unit each
#endif
#define YKA_ITEMS 8                 // macro tiles per unit
#ifndef YKA_TICKETS
#define YKA_TICKETS 4               // tickets a CTA holds ahead of the unit it is issuing
#endif
#ifndef YKA_LAZY_AHEAD
#define YKA_LAZY_AHEAD 1
#endif
#ifndef YKA_LOOKAHEAD
#define YKA_LOOKAHEAD 3
#endif
// YKA_LOOKAHEAD: units the producer may run ahead of the unit the consumers are taking items from
#ifndef YKA_CONS_WARPS
#define YKA_CONS_WARPS 23
#endif
#define YKA_THREADS ((YKA_CONS_WARPS + 1) * 32)
#define YKA_RAW_PLANE_INTS 2272     // 17 rows x 132 ints = 2244, rounded so every plane starts 128-byte aligned
#define YKA_RAW_STAGE_INTS (3 * YKA_RAW_PLANE_INTS + 16 * YK_UNIT_W)
#define YKA_COLOR_TX (3u * YK_RAW_ROWS * YK_RAW_PITCH * 4u)
#define YKA_ALPHA_TX (16u * YK_UNIT_W * 4u)
#define YKA_RAWB_PLANE 2560         // packed upload: 17 rows x 144 bytes = 2448, rounded to a multiple of 128
#define YKA_RAWB_STAGE (3 * YKA_RAWB_PLANE + 16 * YK_UNIT_W)
#define YKA_COLORB_TX (3u * YK_RAW_ROWS * YK_U8_BOX)
#define YKA_ALPHAB_TX (16u * YK_UNIT_W)
#ifndef YKA_PRETEST_CHANNELS
#define YKA_PRETEST_CHANNELS 1
#endif
#ifndef YKA_RANGE_SINGLE
#define YKA_RANGE_SINGLE 0      // 1: the range stage one 8x8 tile at a time (round 1 form, kept for A/B builds)
#endif
#ifndef YKA_STATIC_ROUND_MIN
#define YKA_STATIC_ROUND_MIN 32     // units per CTA from which a launch hands out a whole round of ticket registers statically (a short launch pays for it in its tail)
#endif
#ifndef YKA_PRODUCER_ROLLED
#define YKA_PRODUCER_ROLLED 0
#endif
#ifndef YKA_STATIC_FIRST
#define YKA_STATIC_FIRST 1
#endif
#define YKP_RS 24                   // row pitch in bytes of a warp-private 17x17 byte tile
#define YKP_CH (17 * YKP_RS)        // bytes of one channel of it
#define YKP_TILE 1232               // 3 channels, rounded to a multiple of 16
static_assert(YKA_LOOKAHEAD < YKA_NR, "look-ahead is bounded by the raw ring");

struct YkaUnit {                    // what the producer says about the unit staged in raw buffer i
    int slot, bx, by, k, alpha;     // bx: the first of its two regions
    int seq;                        // which unit of this CTA it is: a consumer checks it before it trusts the barrier's phase parity
};

// the fields of a slot descriptor a consumer warp needs (its own copy, refreshed when its items move to another image)
struct YkaSlotC {
    int slot, w, h, nbx, yOrg, latW, latH, pad;
    const void* rowBelow[3];
    uint32_t* cellMask32;           // claimed cells, two 16-bit rows per word
    uint32_t* touchMap;
    uint8_t*  alphaKept;
    int*      hdr;
    uint32_t* bitmap32[YK_NPASS];
    uint8_t*  latRGB;
    uint8_t*  r2Raw[3];
    uint32_t* r2RawType[3];
};

#define YKA_NSTAT YK_HD_INTS                         // per-pass counters + alpha box / count, laid out like the image header

struct YkaShared {
    uint4    passLane[YK_NPASS][32];    // per pass and lane: see yka_pass_lane_entry
    unsigned long long runTiles;    // bits (of the 41 tiles of a macro tile) of the passes this launch runs
    int      rpOf[8];               // pass id -> its position in the run
    uint8_t  passOfTile[48];        // tile bit -> pass id
    uint32_t pretestTab[41];
    int      queueHead;             // next (unit sequence number * 8 + macro tile) to hand out
    int      endSeq;                // first unit sequence number that does not exist
    int      statSlot;              // the image whose counters are summed in `stat` (other images go straight to global memory)
    int      consLeft;              // consumer warps still running (the last one flushes `stat`)
    int      stat[YKA_NSTAT];
    YkRun    run;
    unsigned long long rawFull[YKA_NR];     // raw buffer i: its TMA boxes have landed
    unsigned long long rawFree[YKA_NR];     // raw buffer i: the four macro tiles of the row have been packed out of it
    YkaUnit  unit[YKA_NR];
};

// everything a consumer warp owns, in one block (one base address serves all of it)
struct alignas(128) YkaWarpArea {
    uint8_t  priv[YKP_TILE];        // the macro tile's 17x17 samples, three channels, as bytes
    uint8_t  hist[768];             // byte counters of the range stage: a 256-byte histogram per half-warp (yka_range_pair), per plane in the single-tile form
    uint32_t touch[28];             // touch words of the 5x5 lattice points of the macro tile
    int      wstat[40];             // 8 groups x 5 counters (see yka_stat_add)
    YkaSlotC slotc;
};

#define YKA_SMEM_RAW   (YKA_NR * YKA_RAW_STAGE_INTS * 4)
#define YKA_SMEM_WARPS (YKA_CONS_WARPS * (int)sizeof(YkaWarpArea))
#define YKA_SMEM_BYTES (YKA_SMEM_RAW + YKA_SMEM_WARPS + 1024 + (int)sizeof(YkaShared))
static_assert(sizeof(YkaWarpArea) % 128 == 0 && YKP_TILE % 16 == 0, "shared-memory carving keeps 128-byte alignment");

// ------------------------------------------------------------------------------------------------------------------
// mbarrier / TMA / shared-flag primitives (inline PTX), with stand-ins for the CPU logic emulation (tests/emu)
#ifdef YK_EMULATE
static inline void yka_mbar_init(unsigned long long* b, int count) { __atomic_store_n(b, (unsigned long long)count << 32, __ATOMIC_SEQ_CST); }
static inline void yka_mbar_expect_tx(unsigned long long*, unsigned) {}
static inline bool yka_mbar_try_wait(unsigned long long* b, unsigned parity) {  // emulated barrier: count << 32 | pending << 16 | completed phases
    if ((__atomic_load_n(b, __ATOMIC_SEQ_CST) & 1ull) != parity) return true;
    std::this_thread::yield();
    return false;
}
static inline void yka_mbar_wait(unsigned long long* b, unsigned parity) { while (!yka_mbar_try_wait(b, parity)) {} }
static inline void yka_mbar_arrive(unsigned long long* b) {
    for (;;) {
        unsigned long long v = __atomic_load_n(b, __ATOMIC_SEQ_CST);
        const unsigned long long count = v >> 32, pending = ((v >> 16) & 0xFFFFull) + 1ull, phases = v & 0xFFFFull;
        const unsigned long long nv = pending == count ? ((count << 32) | ((phases + 1ull) & 0xFFFFull)) : ((count << 32) | (pending << 16) | phases);
        if (__atomic_compare_exchange_n(b, &v, nv, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) return;
    }
}
static inline void yka_tma_box(void* dst, const YkTmap* tm, int x, int y, int bw, int bh, unsigned long long* b, int last) {
    // emulated descriptor: base, width, height, element size, row pitch in elements
    const unsigned char* base = (const unsigned char*)tm->opaque[0];
    const int w = (int)tm->opaque[1], h = (int)tm->opaque[2], es = (int)tm->opaque[3];
    const size_t pitch = (size_t)tm->opaque[4];
    unsigned char* d = (unsigned char*)dst;
    for (int r = 0; r < bh; r++) for (int c = 0; c < bw; c++) {
        if (y + r < h && x + c < w) memcpy(d + ((size_t)r * bw + c) * es, base + ((size_t)(y + r) * pitch + x + c) * es, es);
        else memset(d + ((size_t)r * bw + c) * es, 0, es);
    }
    if (last) yka_mbar_arrive(b);                                               // all boxes of the stage have landed: the phase completes
}
static inline void yka_fence_async() {}
static inline void yka_tmap_acquire(const YkTmap*) {}
static inline int  yka_flag_ld(const int* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline void yka_flag_st(int* p, int v) { __atomic_store_n(p, v, __ATOMIC_SEQ_CST); }
#else
static __device__ __forceinline__ uint32_t yka_s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void yka_mbar_init(unsigned long long* b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(yka_s32(b)), "r"(count) : "memory");
}
static __device__ __forceinline__ void yka_mbar_expect_tx(unsigned long long* b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(yka_s32(b)), "r"(bytes) : "memory");
}
// potentially blocking: the warp is suspended by the hardware until the phase completes or a time limit passes
static __device__ __forceinline__ bool yka_mbar_try_wait(unsigned long long* b, unsigned parity) {
    unsigned ok = 0;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(yka_s32(b)), "r"(parity) : "memory");
    return ok != 0;
}
static __device__ __forceinline__ void yka_mbar_wait(unsigned long long* b, unsigned parity) { while (!yka_mbar_try_wait(b, parity)) {} }
static __device__ __forceinline__ void yka_mbar_arrive(unsigned long long* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(yka_s32(b)) : "memory");
}
static __device__ __forceinline__ void yka_tma_box(void* dst, const YkTmap* tm, int x, int y, int, int, unsigned long long* b, int) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(yka_s32(dst)), "l"((unsigned long long)tm), "r"(x), "r"(y), "r"(yka_s32(b)) : "memory");
}
static __device__ __forceinline__ void yka_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// the descriptors live in global memory and are rewritten by host copies between launches
static __device__ __forceinline__ void yka_tmap_acquire(const YkTmap* tm) {
    asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" :: "l"((unsigned long long)tm) : "memory");
}
// flags in shared memory (LDS / STS, not generic system-scope accesses)
static __device__ __forceinline__ int yka_flag_ld(const int* p) {
    int v; asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(yka_s32(p)) : "memory"); return v;
}
static __device__ __forceinline__ void yka_flag_st(int* p, int v) {
    asm volatile("st.volatile.shared.s32 [%0], %1;" :: "r"(yka_s32(p)), "r"(v) : "memory");
}
#endif

// ------------------------------------------------------------------------------------------------------------------
static __device__ __forceinline__ unsigned yka_pack4(int4 v) {      // low bytes of four samples -> one word (3 PRMT)
    return __byte_perm(__byte_perm((unsigned)v.x, (unsigned)v.y, 0x0040), __byte_perm((unsigned)v.z, (unsigned)v.w, 0x0040), 0x5410);
}
static __device__ __forceinline__ int yka_byte(unsigned word, int k) { return (int)__byte_perm(word, 0u, 0x4440u | (unsigned)k); }

// Lane geometry of one pass, computed once per CTA.  Every lane owns two quads (four consecutive pixels of a row) of
// the macro tile, both inside one tile of the pass:
//   tiles 8 or 16 wide   lane (row = lane >> 1, half = lane & 1): the quads at x = 8*half and 8*half + 4 of that row
//   tiles 4 wide         lane (tx = lane & 3, rp = lane >> 2): the quads at x = 4*tx of rows 2*rp and 2*rp + 1
// (so a pass over 4-wide tiles is one sweep as well).  Entry: x = lanes sharing my tile; y = byte offset of quad 0 | of
// quad 1 << 16 inside a channel of the private tile; z = offset of the tile's top-left sample | the tile's 4x4 cells
// (bit = 4*cellY + cellX) << 16; w = dx0 | dy << 8 | tile index << 16 | leader << 24 (dx0, dy: quad 0 inside the tile).
struct alignas(16) YkaLaneEntry { unsigned x, y, z, w; };
static constexpr YkaLaneEntry yka_pass_lane_entry(int pid, int lane) {
    constexpr int SHX[YK_NPASS] = { 4, 4, 3, 3, 3, 2, 2 }, SHY[YK_NPASS] = { 4, 3, 4, 3, 2, 3, 2 };     // yk_geom_s_tab
    const int shx = SHX[pid], shy = SHY[pid], TW = 1 << shx, TH = 1 << shy;
    int x0 = 0, y0 = 0, x1 = 0, y1 = 0;
    if (shx == 2) { x0 = x1 = 4 * (lane & 3); y0 = 2 * (lane >> 2); y1 = y0 + 1; }
    else { x0 = 8 * (lane & 1); x1 = x0 + 4; y0 = y1 = lane >> 1; }
    const int tx = x0 >> shx, ty = y0 >> shy, lxT = tx << shx, lyT = ty << shy;
    unsigned gmask = 0;
    for (int l = 0; l < 32; l++) {
        const int lx = (shx == 2) ? 4 * (l & 3) : 8 * (l & 1), ly = (shx == 2) ? 2 * (l >> 2) : (l >> 1);
        if ((lx >> shx) == tx && (ly >> shy) == ty) gmask |= 1u << l;
    }
    int first = 0;
    while (!((gmask >> first) & 1u)) first++;
    const int leader = lane == first;
    const unsigned cols = ((1u << (TW >> 2)) - 1u) << (lxT >> 2);
    unsigned cells = 0;
    for (int cy = lyT >> 2; cy < (lyT + TH) >> 2; cy++) cells |= cols << (4 * cy);
    const int t = ty * (16 >> shx) + tx;
    return YkaLaneEntry{ gmask, (unsigned)(y0 * YKP_RS + x0) | ((unsigned)(y1 * YKP_RS + x1) << 16), (unsigned)(lyT * YKP_RS + lxT) | (cells << 16),
                         (unsigned)(x0 - lxT) | ((unsigned)(y0 - lyT) << 8) | ((unsigned)t << 16) | ((unsigned)leader << 24) };
}
// the table, built by the compiler (a CTA copies it to shared memory when it starts: 224 entries that took a 32-step loop each)
struct YkaLaneTable { YkaLaneEntry e[YK_NPASS][32]; };
static constexpr YkaLaneTable yka_make_lane_table() {
    YkaLaneTable t{};
    for (int p = 0; p < YK_NPASS; p++) for (int l = 0; l < 32; l++) t.e[p][l] = yka_pass_lane_entry(p, l);
    return t;
}
__device__ const YkaLaneTable yka_lane_table = yka_make_lane_table();     // global memory: a lane reads its own entry (a constant bank serialises that)

// table entry of tile ti (0..40) of a macro tile: offX | offY << 4 | shx << 8 | shy << 11 | cell << 14
static __device__ __forceinline__ uint32_t yka_pretest_entry(int ti) {
    const int pid = (ti >= 1) + (ti >= 3) + (ti >= 5) + (ti >= 9) + (ti >= 17) + (ti >= 25);
    const int t = ti - (int)((0x19110905030100ull >> (8 * pid)) & 255ull);
    const int shx = (0x2233344 >> (4 * pid)) & 15, shy = (0x2323434 >> (4 * pid)) & 15;
    const int tx = t & ((16 >> shx) - 1), ty = t >> (4 - shx);
    const int offX = tx << shx, offY = ty << shy;
    return (uint32_t)(offX | (offY << 4) | (shx << 8) | (shy << 11) | (((offY >> 2) * 4 + (offX >> 2)) << 14));
}

// per-pass counters / alpha box.  Slot k of a group of five: 0 = count (added), 1..4 = min x, min y (stored as extent -
// value), max x, max y (maxima).  A consumer warp keeps its own sums in shared memory (group p = pass id p, group 7 = the
// alpha stage; lane k owns slot k of every group, so no atomics and no barrier) and adds them to the CTA's sums (or, for
// an image other than the CTA's main one, to the image's header) when its items move to another image and when it retires.
typedef int YkaStat;                // a warp's 8 groups x 5 slots
static __device__ __forceinline__ void yka_stat_add(YkaStat* st, int group, int n, int a, int b, int c, int d) {
    if ((threadIdx.x & 31) == 0) {      // warp-private words: the atomics are fire-and-forget read-modify-writes without contention
        int* p = st + group * 5;
        atomicAdd(&p[0], n); atomicMax(&p[1], a); atomicMax(&p[2], b); atomicMax(&p[3], c); atomicMax(&p[4], d);
    }
}
static __device__ __forceinline__ void yka_stat_flush(YkaShared& sh, const YkaSlotC& C, YkaStat* st) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    if (lane < 8 && st[lane * 5]) {
        const int idx0 = lane < 7 ? YK_HD_PASS0 + lane * YK_ST_STRIDE : YK_HD_ALPHA_KEPT0;
        int* dst = (C.slot == sh.statSlot) ? &sh.stat[idx0] : &C.hdr[idx0];
        atomicAdd(&dst[0], st[lane * 5]);
#pragma unroll
        for (int k = 1; k < 5; k++) atomicMax(&dst[k], st[lane * 5 + k]);
    }
    __syncwarp();
    if (lane < 8) {
#pragma unroll
        for (int k = 0; k < 5; k++) st[lane * 5 + k] = 0;
    }
    __syncwarp();
}

// Consumer warp: its copy of the slot descriptor fields (refreshed when the warp's items move to another image)
static __device__ void yka_slot_refresh(const YkSlotDev& S, YkaSlotC& C, int slot) {
    const int lane = threadIdx.x & 31;
    if (lane == 0) { C.slot = slot; C.w = S.w; C.h = S.h; C.nbx = S.nbx; C.yOrg = S.y0; C.latW = S.latW; C.latH = S.latH; }
    else if (lane == 1) { C.cellMask32 = reinterpret_cast<uint32_t*>(S.cellMask); C.touchMap = S.touchMap; C.alphaKept = S.alphaKept; C.hdr = S.hdr; C.latRGB = S.latRGB; }
    else if (lane >= 2 && lane < 5) { const int p = lane - 2; C.rowBelow[p] = S.rowBelow[p]; C.r2Raw[p] = S.r2Raw[p]; C.r2RawType[p] = S.r2RawType[p]; }
    else if (lane >= 8 && lane < 8 + YK_NPASS) C.bitmap32[lane - 8] = reinterpret_cast<uint32_t*>(S.bitmap[lane - 8]);
    __syncwarp();
}

// all(alpha == 0) of the 16x16 tile of macro tile mx, from the staged alpha rows (samples outside the image arrive as zeros)
template <bool U8>
static __device__ __forceinline__ bool yka_alpha_any(const void* __restrict__ rawv, int mx) {
    const int lane = threadIdx.x & 31;
    bool nz;
    if (U8) {
        const uint2 v = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(rawv) + 3 * YKA_RAWB_PLANE + (lane >> 1) * YK_UNIT_W + 16 * mx + 8 * (lane & 1));
        nz = (v.x | v.y) != 0u;
    } else {
        const int4* __restrict__ a = reinterpret_cast<const int4*>(reinterpret_cast<const int32_t*>(rawv) + 3 * YKA_RAW_PLANE_INTS) + 4 * mx;
        const int4 v0 = a[(lane >> 2) * (YK_UNIT_W / 4) + (lane & 3)], v1 = a[((lane >> 2) + 8) * (YK_UNIT_W / 4) + (lane & 3)];
        nz = (v0.x | v0.y | v0.z | v0.w | v1.x | v1.y | v1.z | v1.w) != 0;
    }
    return __any_sync(YK_FULL, nz);
}

// Consumer warp: the 17x17 samples of macro tile mx (0..7) of the unit whose left edge is X0, three colour planes, from the raw rows
// staged by TMA (int32 samples, or bytes when the image was uploaded packed) into the warp-private byte tile, clamped
// the way Plane::GetPixelValue clamps (framework.h:116-121); then the alpha-zero test of the 16x16 tile (EC.cpp:357-430
// restated per tile).  Returns (uniformly) whether the tile has a non-zero alpha sample.
template <bool U8>
static __device__ __forceinline__ bool yka_pack_macro_tile(const void* __restrict__ rawv, uint8_t* __restrict__ priv, const YkaSlotC& C,
                                                           int X0, int Yk, int mx, bool doAlpha) {
    const int lane = threadIdx.x & 31;
    const int w = C.w, h = C.h;
    const int Xm = X0 + 16 * mx;
    unsigned bad = 0;
    const int32_t* __restrict__ raw = reinterpret_cast<const int32_t*>(rawv);
    const uint8_t* __restrict__ rawb = reinterpret_cast<const uint8_t*>(rawv);
    if (Xm + 20 <= w && Yk + YK_RAW_ROWS <= h) {
        // interior: 17 rows x 20 samples (columns 0..19 of the macro tile, 17 needed) per plane, all inside the image
#pragma unroll
        for (int c = 0; c < 3; c++) {
            uint8_t* __restrict__ d = priv + c * YKP_CH;
#pragma unroll
            for (int it = 0; it < 3; it++) {
                const int idx = it * 32 + lane;                 // 85 = 17 rows x 5 groups of four samples
                if (idx < 85) {
                    const int lr = idx / 5, q = idx - lr * 5;
                    unsigned packed;
                    if (U8) {
                        packed = *reinterpret_cast<const unsigned*>(rawb + c * YKA_RAWB_PLANE + lr * YK_U8_BOX + 16 * mx + 4 * q);
                    } else {
                        const int4 v = (reinterpret_cast<const int4*>(raw + c * YKA_RAW_PLANE_INTS) + 4 * mx)[lr * (YK_RAW_PITCH / 4) + q];
                        bad |= (unsigned)(v.x | v.y | v.z | v.w);
                        packed = yka_pack4(v);
                    }
                    *reinterpret_cast<unsigned*>(d + lr * YKP_RS + 4 * q) = packed;
                }
            }
        }
    } else if (Yk < h && Xm < w) {
        // at the right / bottom edge: clamp inside the image; in strip mode the row under the strip is the real image
        // row (rowBelow), not a clamp
        const int wmax = w - 1 - X0, hmax = min(16, h - 1 - Yk);
        for (int idx = lane; idx < 17 * 17; idx += 32) {
            const int lr = idx / 17, lx = idx - lr * 17;
#pragma unroll
            for (int c = 0; c < 3; c++) {
                int s;
                if (lr > hmax && C.rowBelow[c]) {
                    const int x = min(Xm + lx, w - 1);
                    s = U8 ? (int)__ldg(reinterpret_cast<const uint8_t*>(C.rowBelow[c]) + x) : __ldg(reinterpret_cast<const int32_t*>(C.rowBelow[c]) + x);
                } else {
                    const int rr = min(lr, hmax), cc = min(16 * mx + lx, wmax);
                    s = U8 ? (int)rawb[c * YKA_RAWB_PLANE + rr * YK_U8_BOX + cc] : raw[c * YKA_RAW_PLANE_INTS + rr * YK_RAW_PITCH + cc];
                }
                bad |= (unsigned)s;
                priv[c * YKP_CH + lr * YKP_RS + lx] = (uint8_t)s;
            }
        }
    }
    if (bad & ~255u) atomicOr(&C.hdr[YK_HD_ERR], 1);
    bool kept = false;
    if (doAlpha) kept = yka_alpha_any<U8>(rawv, mx);
    return kept;
}

// ------------------------------------------------------------------------------------------------------------------
// Cheap rejection of all 41 tiles (1 + 2 + 2 + 4 + 8 + 8 + 16 over the seven shapes) of a 16x16 macro tile: lane = tile,
// the quad at the tile centre of every channel, raw corners.  A pixel whose raw-family U is outside [loWide, hiWide) cannot
// be accepted by any of the six variants (a family's corners differ from the raw ones by -3..+4), so a cleared bit is a
// proven rejection; a set bit only means "run the real test".  Bit (start(pid) + t) belongs to tile t of pass id pid.
static __device__ __forceinline__ unsigned long long yka_pretest(const uint8_t* __restrict__ priv, const uint32_t* sTab, int wIn, int hIn,
                                                                 unsigned claimed, int R) {
    const int lane = threadIdx.x & 31;
    unsigned long long P = 0;
#pragma unroll
    for (int round = 0; round < 2; round++) {
        const int ti = lane + 32 * round;
        bool possible = false;
        if (ti < 41) {
            const uint32_t e = sTab[ti];
            const int shx = (e >> 8) & 7, shy = (e >> 11) & 7, sh = shx + shy;
            const int lx0 = e & 15, ly0 = (e >> 4) & 15, TW = 1 << shx, TH = 1 << shy, N = 1 << sh;
            if (!((claimed >> (e >> 14)) & 1u) && lx0 + TW <= wIn && ly0 + TH <= hIn) {
                const int dx0 = (TW >> 1) & ~3, dy = TH >> 1;
                const int loW = -(4 * N + N / 2 - 1), hiW = (2 * R + 4) * N;
                possible = true;
#pragma unroll
                for (int c = 0; c < YKA_PRETEST_CHANNELS; c++) {
                    const uint8_t* p = priv + c * YKP_CH + ly0 * YKP_RS + lx0;
                    const int tl = p[0], tr = p[TW], bl = p[TH * YKP_RS], br = p[TH * YKP_RS + TW];
                    const unsigned word = *reinterpret_cast<const unsigned*>(p + dy * YKP_RS + dx0);
                    const int B = (tr - tl) << shy, C = (bl - tl) << shx, D = tl - tr - bl + br;
                    const int step = B + D * dy;
                    const int s0 = ((tl + R) << sh) + B * dx0 + dy * (C + D * dx0);
                    const int u0 = s0 - (int)((word & 255u) << sh), u1 = s0 + step - (int)(((word >> 8) & 255u) << sh);
                    const int u2 = s0 + 2 * step - (int)(((word >> 16) & 255u) << sh), u3 = s0 + 3 * step - (int)((word >> 24) << sh);
                    const int umin = __vimin3_s32(min(u0, u1), u2, u3), umax = __vimax3_s32(max(u0, u1), u2, u3);
                    possible = possible && !(umin < loW || umax >= hiW);
                }
            }
        }
        P |= (unsigned long long)__ballot_sync(YK_FULL, possible) << (32 * round);
    }
    return P;
}

// four consecutive pixels of one channel: U = S + R*N - cur*N folded into a running min/max.
// |cur - S/N| <= R  <=>  0 <= U < (2R+1)N;   |cur - (S+N/2-1)/N| <= R  <=>  -(N/2-1) <= U < (2R+1)N-(N/2-1)
// (S = bilinear numerator with integer weights; identical to ((bT*tF+bB*bF)[+2^19-1])>>20 of EC.cpp:3937-3965).
static __device__ __forceinline__ void yka_quad(unsigned word, int s, int step, int negN, int& umin, int& umax) {
    const int s1 = s + step, s2 = s1 + step, s3 = s2 + step;
    const int u0 = yka_byte(word, 0) * negN + s;
    const int u1 = yka_byte(word, 1) * negN + s1;
    const int u2 = yka_byte(word, 2) * negN + s2;
    const int u3 = yka_byte(word, 3) * negN + s3;
    umin = __vimin3_s32(umin, u0, u1); umin = __vimin3_s32(umin, u2, u3);
    umax = __vimax3_s32(umax, u0, u1); umax = __vimax3_s32(umax, u2, u3);
}

struct YkaTile {                    // per lane: the tile it belongs to in the current pass
    int shx, shy, sh, negN, dx0, dy, R;
    bool wide;                      // tiles 8 or 16 wide: quad 1 continues the row of quad 0; 4 wide: it is the quad below
};

// one channel of one corner family: this lane's two quads against the bilinear fit of (tl, tr, bl, br)
static __device__ __forceinline__ void yka_channel(const YkaTile& T, unsigned w0, unsigned w1, int tl, int tr, int bl, int br, int& umin, int& umax) {
    const int B = (tr - tl) << T.shy, C = (bl - tl) << T.shx, D = tl - tr - bl + br;
    const int step = B + D * T.dy, down = C + D * T.dx0;
    const int s = ((tl + T.R) << T.sh) + B * T.dx0 + T.dy * down;
    yka_quad(w0, s, step, T.negN, umin, umax);
    yka_quad(w1, T.wide ? s + 4 * step : s + down, T.wide ? step : step + D, T.negN, umin, umax);
}

// The accept test of FittingQuadSmooth (EC.cpp:3810-3998) for the tile this lane belongs to.  The lanes in `gmask` share
// the tile; each holds two quads of it (w0 / w1 per channel, see yka_pass_lane_entry).
// Returns, uniformly over the group, whether any of the six variants (3 corner families x rounded / truncated) keeps
// every pixel of every channel within the reject factor.
static __device__ __forceinline__ bool yka_tile_test(const uint8_t* __restrict__ corner, const YkaTile& T, const unsigned (&w0)[3], const unsigned (&w1)[3],
                                                     unsigned gmask, bool active) {
    const int N = 1 << T.sh, TW = 1 << T.shx, THp = YKP_RS << T.shy;
    const int hiT = (2 * T.R + 1) * N;                  // |cur - S/N| <= R            <=>  0 <= U < hiT
    const int loR = -(N / 2 - 1);                       // |cur - (S+N/2-1)/N| <= R    <=>  loR <= U < hiT + loR
    const int loWide = -(4 * N + N / 2 - 1), hiWide = hiT + 3 * N;
    int cr[3][4];                                       // TL TR BL BR, clamped at the image edge by the packing (EC.cpp:3845-3868)
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const uint8_t* p = corner + c * YKP_CH;
        cr[c][0] = p[0]; cr[c][1] = p[TW]; cr[c][2] = p[THp]; cr[c][3] = p[THp + TW];
    }
    bool resolved = !active;
    // ---- raw corners
    int umin = INT_MAX, umax = INT_MIN;
    yka_channel(T, w0[0], w1[0], cr[0][0], cr[0][1], cr[0][2], cr[0][3], umin, umax);
    {   // one channel with the raw corners proves most non-gradient tiles hopeless for every variant
        const unsigned bH = __ballot_sync(YK_FULL, (umin < loWide) || (umax >= hiWide));
        if (bH & gmask) resolved = true;
        if (!__any_sync(YK_FULL, !resolved)) return false;
    }
    yka_channel(T, w0[1], w1[1], cr[1][0], cr[1][1], cr[1][2], cr[1][3], umin, umax);
    yka_channel(T, w0[2], w1[2], cr[2][0], cr[2][1], cr[2][2], cr[2][3], umin, umax);
    const unsigned bT = __ballot_sync(YK_FULL, (umin < 0) || (umax >= hiT));
    const unsigned bR = __ballot_sync(YK_FULL, (umin < loR) || (umax >= hiT + loR));
    const unsigned bH = __ballot_sync(YK_FULL, (umin < loWide) || (umax >= hiWide));
    bool accepted = !resolved && (((bT & gmask) == 0u) || ((bR & gmask) == 0u));     // EC.cpp:3998: any surviving variant accepts
    if (accepted || (bH & gmask)) resolved = true;                                   // no family can accept a tile outside the wide bounds
    if (!__any_sync(YK_FULL, !resolved)) return accepted;
    // ---- Round6 corners
    {
        int umin1 = INT_MAX, umax1 = INT_MIN;
#pragma unroll
        for (int c = 0; c < 3; c++)
            yka_channel(T, w0[c], w1[c], yk_round6(cr[c][0]), yk_round6(cr[c][1]), yk_round6(cr[c][2]), yk_round6(cr[c][3]), umin1, umax1);
        const unsigned bT1 = __ballot_sync(YK_FULL, (umin1 < 0) || (umax1 >= hiT));
        const unsigned bR1 = __ballot_sync(YK_FULL, (umin1 < loR) || (umax1 >= hiT + loR));
        if (!resolved && (((bT1 & gmask) == 0u) || ((bR1 & gmask) == 0u))) { accepted = true; resolved = true; }
        if (!__any_sync(YK_FULL, !resolved)) return accepted;
    }
    // ---- Round6P corners
    {
        int umin2 = INT_MAX, umax2 = INT_MIN;
#pragma unroll
        for (int c = 0; c < 3; c++)
            yka_channel(T, w0[c], w1[c], yk_round6p(cr[c][0]), yk_round6p(cr[c][1]), yk_round6p(cr[c][2]), yk_round6p(cr[c][3]), umin2, umax2);
        const unsigned bT2 = __ballot_sync(YK_FULL, (umin2 < 0) || (umax2 >= hiT));
        const unsigned bR2 = __ballot_sync(YK_FULL, (umin2 < loR) || (umax2 >= hiT + loR));
        if (!resolved && (((bT2 & gmask) == 0u) || ((bR2 & gmask) == 0u))) accepted = true;
    }
    return accepted;
}

// Side effects of an accepted tile (EC.cpp:3998-4132) other than its counters: bitmap bit, the four lattice points it
// touches with its role at each.  (gx0, gy0) = tile origin in the image, (tlx, tly) = inside the macro tile.
static __device__ __forceinline__ void yka_commit(const YkaSlotC& C, uint32_t* __restrict__ touch, const YkGeomS& g, int pid, int rp,
                                                  int gx0, int gy0, int tlx, int tly) {
    const int TW = 1 << g.shx, TH = 1 << g.shy;
    const int nSwzX = (C.w + (1 << g.lbw) - 1) >> g.lbw;
    const int pos = yk_pos_s(g, nSwzX, gx0 >> g.shx, gy0 >> g.shy);
    atomicOr(&C.bitmap32[pid][pos >> 5], 1u << (pos & 31));                    // EC.cpp:4026
    const int i0 = tlx >> 2, j0 = tly >> 2;                                    // mappedRGB claim, EC.cpp:4001-4021
    atomicOr(&touch[j0 * 5 + i0], 1u << (4 * rp + 0));
    atomicOr(&touch[j0 * 5 + i0 + (TW >> 2)], 1u << (4 * rp + 1));
    atomicOr(&touch[(j0 + (TH >> 2)) * 5 + i0], 1u << (4 * rp + 2));
    atomicOr(&touch[(j0 + (TH >> 2)) * 5 + i0 + (TW >> 2)], 1u << (4 * rp + 3));
}

// One FittingQuadSmooth pass over one 16x16 macro tile, by one warp, all tiles of the pass in one sweep (lane geometry:
// yka_pass_lane_entry).  `poss`: the tiles to test (eligible - EC.cpp:3818, 3826, 3871-3875 - and not proven hopeless).
// Returns (uniformly) the cells the accepted tiles claim (16 bits, bit = 4*cellY + cellX) and counts them in `st`.
static __device__ __forceinline__ unsigned yka_macro_pass(const uint8_t* __restrict__ priv, const YkaShared& sh, const YkaSlotC& C, uint32_t* __restrict__ touch,
                                                          YkaStat* st, int pid, int gmx, int gmy, unsigned poss, int rej) {
    const YkGeomS g = yk_geom_s(pid);
    const int lane = threadIdx.x & 31;
    const uint4 e = sh.passLane[pid][lane];
    YkaTile T;
    T.shx = g.shx; T.shy = g.shy; T.sh = g.shx + g.shy; T.negN = -(1 << T.sh); T.R = rej; T.wide = g.shx != 2;
    T.dx0 = e.w & 255u; T.dy = (e.w >> 8) & 255u;
    const bool active = (poss >> ((e.w >> 16) & 255u)) & 1u;
    unsigned w0[3], w1[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        w0[c] = *reinterpret_cast<const unsigned*>(priv + c * YKP_CH + (e.y & 0xFFFFu));
        w1[c] = *reinterpret_cast<const unsigned*>(priv + c * YKP_CH + (e.y >> 16));
    }
    const int cornerOff = e.z & 0xFFFFu;
    const bool acc = yka_tile_test(priv + cornerOff, T, w0, w1, e.x, active);
    const bool mineAcc = acc && (e.w >> 24);
    const unsigned accB = __ballot_sync(YK_FULL, mineAcc);
    if (!accB) return 0u;
    if (mineAcc) {
        const int tly = cornerOff / YKP_RS, tlx = cornerOff - tly * YKP_RS;
        yka_commit(C, touch, g, pid, sh.rpOf[pid], gmx + tlx, gmy + tly, tlx, tly);
    }
    const unsigned cells = __reduce_or_sync(YK_FULL, mineAcc ? (e.z >> 16) : 0u);          // EC.cpp:4029-4037
    // TileDone and the bounding box of the accepted tiles (EC.cpp:4039-4044) from the cells they cover
    const unsigned colm = (cells | (cells >> 4) | (cells >> 8) | (cells >> 12)) & 15u;
    const unsigned rowm = ((cells & 0x000Fu) ? 1u : 0u) | ((cells & 0x00F0u) ? 2u : 0u) | ((cells & 0x0F00u) ? 4u : 0u) | ((cells & 0xF000u) ? 8u : 0u);
    const int x0 = gmx + 4 * (__ffs((int)colm) - 1), x1 = gmx + 4 * (32 - __clz((int)colm));
    const int y0 = gmy + 4 * (__ffs((int)rowm) - 1), y1 = gmy + 4 * (32 - __clz((int)rowm));
    yka_stat_add(st, pid, __popc(accB), C.w - x0, INT_MAX / 2 - (C.yOrg + y0), x1, C.yOrg + y1);
    return cells;
}

// Tiles (bits as in the pre-test: start(pid) + t) whose top-left cell is unclaimed (EC.cpp:3871-3875), from the claimed
// cells of the macro tile (bit = 4*cellY + cellX).  Warp-uniform bit arithmetic.
static __device__ __forceinline__ unsigned long long yka_eligible(unsigned claimed) {
    const unsigned f = ~claimed & 0xFFFFu;
    unsigned e = f & 0x5555u;                           // cells with even x, compressed: bit i = cell 2*i
    e = (e | (e >> 1)) & 0x3333u; e = (e | (e >> 2)) & 0x0F0Fu; e = (e | (e >> 4)) & 0x00FFu;
    const unsigned lo = (f & 1u)                                              // 16x16: cell 0
                      | (((e & 1u) | ((e >> 3) & 2u)) << 1)                   // 16x8: cells 0, 8
                      | ((e & 3u) << 3)                                       // 8x16: cells 0, 2
                      | (((e & 3u) | ((e >> 2) & 12u)) << 5)                  // 8x8: cells 0, 2, 8, 10
                      | (e << 9)                                              // 8x4: cells 0, 2, .. 14
                      | (((f & 15u) | ((f >> 4) & 0xF0u)) << 17);             // 4x8: cells 0..3, 8..11
    return (unsigned long long)lo | ((unsigned long long)f << 25);           // 4x4: every cell
}

#if YKA_RANGE_SINGLE     // the round 1 form, one 8x8 tile at a time: kept for A/B builds (tools/ab_build.py)
// DynamicTileCompressor (EC.cpp:8398-8522) for the 8x8 tile at (lx8, ly8) of the macro tile; q = its quadrants to code
// (bit0 TL, 1 TR, 2 BL, 3 BR: top-left map pixel 0, EC.cpp:8420-8430 == 4x4 cell unclaimed).  Lane = two pixels; the
// three planes side by side.  Output goes to the tile's fixed place in r2Raw / r2RawType.
static __device__ __forceinline__ void yka_range_tile(const uint8_t* __restrict__ priv, const YkaSlotC& Rg, uint8_t* __restrict__ hist,
                                                      const uint32_t* __restrict__ magicTab, size_t tile, int lx8, int ly8, unsigned q) {
    const int lane = threadIdx.x & 31;
    const int r = lane >> 2, c0 = (lane & 3) * 2;           // pixel row / first column of this lane inside the tile
    const int band = r >> 2, right = c0 >> 2;
    const bool valid = (q >> (band * 2 + right)) & 1u;
    const unsigned qb = (q >> (band * 2)) & 3u;             // coded quadrants of this band: bit0 left, bit1 right
    const int lengthX = (qb == 3u) ? 8 : 4, x2 = (qb == 2u) ? 4 : 0;
    const int pos = (band ? 16 * __popc(q & 3u) : 0) + (r & 3) * lengthX + (c0 - x2);
    // One plane at a time, the loop NOT unrolled: the side-by-side form (three planes interleaved) was 370 instructions
    // against 130 and 10 % slower for the whole kernel - the consumers' code has to stay small (instruction cache).
    // FindAndRemoveMostUsedColor (EC.cpp:8335-8356): per-value counts in a byte histogram (four 8-bit counters per word,
    // a tile has at most 64 pixels), filled with shared-memory atomics
    uint32_t* hist32 = reinterpret_cast<uint32_t*>(hist);
#pragma unroll 1
    for (int p = 0; p < 3; p++) {
        const unsigned short two = *reinterpret_cast<const unsigned short*>(priv + p * YKP_CH + (ly8 + r) * YKP_RS + lx8 + c0);
        const int vx = two & 255, vy = two >> 8;             // CompressF(v,255) == v (EC.cpp:8442)
        uint8_t* hp = hist + p * 256;
        if (valid) {
            atomicAdd(&hist32[p * 64 + (vx >> 2)], 1u << (8 * (vx & 3)));
            atomicAdd(&hist32[p * 64 + (vy >> 2)], 1u << (8 * (vy & 3)));
        }
        __syncwarp();
        // highest index among the maximal counts (`>=`, EC.cpp:8340); only present values can win
        unsigned key = valid ? max(((unsigned)hp[vx] << 8) | (unsigned)vx, ((unsigned)hp[vy] << 8) | (unsigned)vy) : 0u;
        key = __reduce_max_sync(YK_FULL, key);
        if (valid) { hp[vx] = 0; hp[vy] = 0; }               // clean again for the next tile (ordered by the reductions below)
        const int color0 = min(max((int)(key & 255u), 1), 254);
        // Model1 (EC.cpp:8358-8381) over what is left of the histogram
        const bool remx = valid && (vx < color0 - 1 || vx > color0 + 1);
        const bool remy = valid && (vy < color0 - 1 || vy > color0 + 1);
        const int mn = __reduce_min_sync(YK_FULL, min(remx ? vx : 999, remy ? vy : 999));
        const int mx = __reduce_max_sync(YK_FULL, max(remx ? vx : -1, remy ? vy : -1));
        int minCol = 0, delta = 0;
        if (mn != 999) { minCol = mn; delta = mx - mn; }
        if (valid) {
            // GetValueModel1 (EC.cpp:8383-8391): C division of a numerator in -1..3951 by delta in 1..255.
            // floor(n/d) == (n * ceil(2^20/d)) >> 20 for 0 <= n < 4112, d <= 255; n == -1 only happens for delta == 1.
            int bxv = 0, byv = 0;
            if (delta) {
                const unsigned magic = magicTab[delta];
                const int rnd = (delta >> 1) - 1;
                if (remx) { const int n = (vx - minCol) * 15 + rnd; bxv = 1 + (n < 0 ? n : (int)(((unsigned)n * magic) >> 20)); }
                if (remy) { const int n = (vy - minCol) * 15 + rnd; byv = 1 + (n < 0 ? n : (int)(((unsigned)n * magic) >> 20)); }
            } else { bxv = remx ? 1 : 0; byv = remy ? 1 : 0; }
            *reinterpret_cast<uint16_t*>(Rg.r2Raw[p] + tile * 64 + pos) = (uint16_t)((bxv & 255) | ((byv & 255) << 8));
        }
        if (lane == 0) Rg.r2RawType[p][tile] = (uint32_t)color0 | ((uint32_t)minCol << 8) | ((uint32_t)delta << 16);     // EC.cpp:8503-8505
    }
    __syncwarp();       // the histogram entries are clean again before the next tile fills them
}
#endif

// maximum over the lanes of the caller's half-warp.  Two full-warp reductions: a reduction whose member mask differs between
// the lanes of a warp is compiled into a divergent path (WARPSYNC.COLLECTIVE per mask) that leaves the halves running apart.
static __device__ __forceinline__ unsigned yka_half_max(unsigned v, int upper) {
    const unsigned a = __reduce_max_sync(YK_FULL, upper ? 0u : v), b = __reduce_max_sync(YK_FULL, upper ? v : 0u);
    return upper ? b : a;
}

// The same for the two 8x8 tiles of one half (upper / lower) of the macro tile at once: half-warp h codes the tile at
// (8*h, ly8), a lane four consecutive pixels of a row - exactly one row of one 4x4 cell, so a lane is coded or not as a
// whole and its four index bytes are one aligned word of the tile's compact output.  Per value the count comes back from
// the shared-memory atomic itself (the last lane to add a value sees its count - 1, so the maximum of old << 8 | value
// over the lanes is the most used value, highest index among equals: EC.cpp:8340) - no second look at the histogram;
// the reductions run per half-warp (yka_half_max).  qL / qR: quadrants to code of the left / right tile.
static __device__ __forceinline__ void yka_range_pair(const uint8_t* __restrict__ priv, const YkaSlotC& Rg, uint8_t* __restrict__ hist,
                                                      const uint32_t* __restrict__ magicTab, size_t tileL, int ly8, unsigned qL, unsigned qR) {
    const int lane = threadIdx.x & 31;
    const int h = lane >> 4, l = lane & 15, r = l >> 1, right = l & 1;
    const unsigned q = h ? qR : qL;
    const int band = r >> 2;
    const bool valid = (q >> (band * 2 + right)) & 1u;
    const unsigned qb = (q >> (band * 2)) & 3u;             // coded quadrants of this band: bit0 left, bit1 right
    const int lengthX = (qb == 3u) ? 8 : 4, x2 = (qb == 2u) ? 4 : 0;
    const int pos = (band ? 16 * __popc(q & 3u) : 0) + (r & 3) * lengthX + (4 * right - x2);
    const size_t tile = tileL + h;
    uint32_t* hw = reinterpret_cast<uint32_t*>(hist) + 64 * h;              // byte counters, four to a word; one histogram per half-warp
    const uint8_t* src = priv + (ly8 + r) * YKP_RS + 8 * h + 4 * right;
#pragma unroll 1
    for (int p = 0; p < 3; p++) {
        const unsigned word = *reinterpret_cast<const unsigned*>(src + p * YKP_CH);      // CompressF(v,255) == v (EC.cpp:8442)
        int v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) v[k] = yka_byte(word, k);
        // FindAndRemoveMostUsedColor (EC.cpp:8335-8356)
        unsigned key = 0;
        if (valid) {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const unsigned s8 = (unsigned)(v[k] & 3) * 8u - 8u;                         // rotations take it modulo 32
                const unsigned old = atomicAdd(&hw[v[k] >> 2], __funnelshift_l(0x100u, 0x100u, s8));
                key = max(key, (__funnelshift_r(old, old, s8) & 0xFF00u) | (unsigned)v[k]);
            }
        }
        key = yka_half_max(key, h);
        reinterpret_cast<uint4*>(hw)[l] = make_uint4(0u, 0u, 0u, 0u);                       // clean again (every add came back before the reduction)
        const int color0 = min(max((int)(key & 255u), 1), 254);
        // Model1 (EC.cpp:8358-8381) over what is left of the histogram
        bool rem[4];
        unsigned lo = 999u, hi = 0u;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            rem[k] = valid && (unsigned)(v[k] - (color0 - 1)) > 2u;
            lo = min(lo, rem[k] ? (unsigned)v[k] : 999u);
            hi = max(hi, rem[k] ? (unsigned)v[k] : 0u);
        }
        const unsigned mn = 999u - yka_half_max(999u - lo, h);
        const unsigned mx = yka_half_max(hi, h);
        int minCol = 0, delta = 0;
        if (mn != 999u) { minCol = (int)mn; delta = (int)(mx - mn); }
        // GetValueModel1 (EC.cpp:8383-8391): 1 + n / delta (C division), n = (v - minCol) * 15 + delta / 2 - 1 >= -1, is
        // floor((n + delta) / delta) = ((2 * (n + delta)) * (ceil(2^22 / delta) << 9)) >> 32, exact for n + delta < 16448;
        // delta == 0 (every remaining pixel == minCol) gives 1: the table holds 2^31 for it and the numerator is 2
        const int K = delta ? 2 * ((delta >> 1) - 1 + delta - 15 * minCol) : 2 - 30 * minCol;
        const unsigned magic = magicTab[delta];
        if (valid) {
            unsigned b[4];
#pragma unroll
            for (int k = 0; k < 4; k++) b[k] = rem[k] ? __umulhi((unsigned)(v[k] * 30 + K), magic) : 0u;
            *reinterpret_cast<uint32_t*>(Rg.r2Raw[p] + tile * 64 + pos) = __byte_perm(__byte_perm(b[0], b[1], 0x0040), __byte_perm(b[2], b[3], 0x0040), 0x5410);
        }
        if (l == 0 && q) Rg.r2RawType[p][tile] = (uint32_t)color0 | ((uint32_t)minCol << 8) | ((uint32_t)delta << 16);     // EC.cpp:8503-8505
        __syncwarp();       // the cleared counters are in place before the next plane's adds
    }
}


template <bool U8>
static __device__ __forceinline__ int yka_pass16_raw(const void* __restrict__ rawv, const YkaSlotC& C, YkaStat* st, int gmx, int gmy, int mx, int R) {
    const int lane = threadIdx.x & 31, row = lane >> 1, half = lane & 1;
    constexpr int N = 256;
    const int hiT = (2 * R + 1) * N, loR = -(N / 2 - 1), loWide = -(4 * N + N / 2 - 1), hiWide = hiT + 3 * N;
    int umin = INT_MAX, umax = INT_MIN;
    unsigned bad = 0;
    int corner[3];                                       // TL of each channel (what the macro tile's own lattice point emits)
#pragma unroll
    for (int c = 0; c < 3; c++) {
        int tl, tr, bl, br, v[8];
        if (U8) {
            const uint8_t* p = reinterpret_cast<const uint8_t*>(rawv) + c * YKA_RAWB_PLANE + 16 * mx;
            tl = p[0]; tr = p[16]; bl = p[16 * YK_U8_BOX]; br = p[16 * YK_U8_BOX + 16];
            const uint2 w = *reinterpret_cast<const uint2*>(p + row * YK_U8_BOX + 8 * half);
#pragma unroll
            for (int k = 0; k < 4; k++) { v[k] = yka_byte(w.x, k); v[4 + k] = yka_byte(w.y, k); }
        } else {
            const int32_t* p = reinterpret_cast<const int32_t*>(rawv) + c * YKA_RAW_PLANE_INTS + 16 * mx;
            tl = p[0]; tr = p[16]; bl = p[16 * YK_RAW_PITCH]; br = p[16 * YK_RAW_PITCH + 16];
            const int4 a = *reinterpret_cast<const int4*>(p + row * YK_RAW_PITCH + 8 * half), b = *reinterpret_cast<const int4*>(p + row * YK_RAW_PITCH + 8 * half + 4);
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
            bad |= (unsigned)(a.x | a.y | a.z | a.w | b.x | b.y | b.z | b.w | tr | bl | br);
        }
        corner[c] = tl;
        const int B = (tr - tl) * 16, Cc = (bl - tl) * 16, D = tl - tr - bl + br;
        const int step = B + D * row;
        int sk = (tl + R) * N + B * (8 * half) + row * (Cc + D * (8 * half));
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const int u0 = sk - v[k] * N, u1 = sk + step - v[k + 1] * N;
            umin = __vimin3_s32(umin, u0, u1); umax = __vimax3_s32(umax, u0, u1);
            sk += 2 * step;
        }
        if (c == 0 && __any_sync(YK_FULL, (umin < loWide) || (umax >= hiWide))) return 2;     // warp-uniform
    }
    if (bad & ~255u) atomicOr(&C.hdr[YK_HD_ERR], 1);
    const bool dT = __any_sync(YK_FULL, (umin < 0) || (umax >= hiT));
    const bool dR = __any_sync(YK_FULL, (umin < loR) || (umax >= hiT + loR));
    if (dT && dR) return __any_sync(YK_FULL, (umin < loWide) || (umax >= hiWide)) ? 2 : 0;
    // ---- accepted (EC.cpp:3998-4132): bitmap bit, counters, claimed cells, the four touched lattice points, corner colours
    const YkGeomS g = yk_geom_s(0);
    if (lane == 0) {
        const int nSwzX = (C.w + 63) >> 6;
        const int pos = yk_pos_s(g, nSwzX, gmx >> 4, gmy >> 4);
        atomicOr(&C.bitmap32[0][pos >> 5], 1u << (pos & 31));
    }
    yka_stat_add(st, 0, 1, C.w - gmx, INT_MAX / 2 - (C.yOrg + gmy), gmx + 16, C.yOrg + gmy + 16);
    const int cx0 = gmx >> 2, cy0 = gmy >> 2;
    if (lane < 4) {
        const int e = (cy0 + lane) * C.nbx + (cx0 >> 4);
        atomicOr(&C.cellMask32[e >> 1], 15u << (16 * (e & 1) + (cx0 & 15)));
        // pass position 0: corner role k of the tile at its lattice point k (TL, TR, BL, BR)
        atomicOr(&C.touchMap[(size_t)(cy0 + 4 * (lane >> 1)) * C.latW + cx0 + 4 * (lane & 1)], 1u << lane);
    }
    return 1;
}

#ifdef YK_TIMING
__device__ unsigned long long yk_timing[32];
static __device__ __forceinline__ unsigned long long ykt_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define YKT_DECL long long t__ = clock64(), t2__
#define YKT(i) (t2__ = clock64(), atomicAdd(&yk_timing[i], (unsigned long long)(t2__ - t__)), t__ = t2__)
extern "C" void yk_debug_timing(unsigned long long* out, int reset) {
    cudaMemcpyFromSymbol(out, yk_timing, sizeof(yk_timing));
    if (reset) { unsigned long long z[32] = {0}; cudaMemcpyToSymbol(yk_timing, z, sizeof(z)); }
}
#else
#define YKT_DECL
#define YKT(i)
#endif

// One macro tile after its pixels have been packed: the cascade of Convert()'s passes (EC.cpp:9057-9093), its results,
// the corner colours of its lattice points, then the range stage.  (gmx, gmy) = origin of the macro tile in the image.
static __device__ __forceinline__ void yka_macro_tile(const uint8_t* __restrict__ priv, YkaShared& sh, const YkaSlotC& C, uint32_t* __restrict__ touch, uint8_t* hist,
                                      const uint32_t* magicTab, YkaStat* st, int gmx, int gmy, bool pass16Hopeless) {
    const int lane = threadIdx.x & 31;
    const YkRun& run = sh.run;
    YKT_DECL;
    const int wIn = C.w - gmx, hIn = C.h - gmy;              // image extent seen from the macro tile's origin
    if (wIn <= 0 || hIn <= 0) return;
    // claimed 4x4 cells of the macro tile (bit = 4*cellY + cellX); cells outside the image count as claimed
    unsigned claimed = 0;
    const int cx0 = gmx >> 2, cy0 = gmy >> 2, cellWord = cx0 >> 4, cellShift = cx0 & 15;
    if (!run.fresh) {
        unsigned rowBits = 0;
        if (lane < 4 && 4 * lane < hIn) {
            const int e = (cy0 + lane) * C.nbx + cellWord;
            rowBits = ((__ldg(&C.cellMask32[e >> 1]) >> (16 * (e & 1) + cellShift)) & 15u) << (4 * lane);
        }
        claimed = __reduce_or_sync(YK_FULL, rowBits);
    }
    {
        const int cw = min(4, wIn >> 2), chh = min(4, hIn >> 2);
        const unsigned inside = (((1u << cw) - 1u) * 0x1111u) & ((1u << (4 * chh)) - 1u);
        claimed |= ~inside & 0xFFFFu;
    }
    const unsigned claimed0 = claimed;
    if (run.nPasses > 0) {
        if (lane < 25) touch[lane] = 0;
        __syncwarp();
        if (claimed != 0xFFFFu) {
            // All 41 tiles of the seven shapes are pre-tested together; `todo` = the tiles of the run's passes that are
            // inside the image, eligible and not proven hopeless.  The passes run in Convert()'s order = bit order, and only
            // those that still have a tile to test; a pass that accepts tiles makes the tiles under them ineligible.
            const int rej = run.rejectFactor;
            unsigned long long todo = yka_pretest(priv, sh.pretestTab, wIn, hIn, claimed, rej) & sh.runTiles;
            if (pass16Hopeless) todo &= ~1ull;
            while (todo) {
                const int pid = sh.passOfTile[__ffsll((long long)todo) - 1];
                const YkGeomS g = yk_geom_s(pid);
                const int nT = 256 >> (g.shx + g.shy);
                const unsigned poss = (unsigned)(todo >> g.start) & ((1u << nT) - 1u);
                todo &= ~0ull << (g.start + nT);
                const unsigned cells = yka_macro_pass(priv, sh, C, touch, st, pid, gmx, gmy, poss, rej);
                if (cells) { claimed |= cells; todo &= yka_eligible(claimed); }
            }
            if (threadIdx.x == 32) YKT(11);
            // EC.cpp:4029-4037: newly claimed cells
            const unsigned fresh4 = ((claimed & ~claimed0) >> (4 * (lane & 3))) & 15u;
            if (lane < 4 && fresh4) {
                const int e = (cy0 + lane) * C.nbx + cellWord;
                atomicOr(&C.cellMask32[e >> 1], fresh4 << (16 * (e & 1) + cellShift));
            }
        }
        __syncwarp();
        if (lane < 25) {
            // the macro tile's 5x5 lattice points: their touch words, and the corner colour an accepted tile would emit
            // there (EC.cpp:4115-4132); the points on the right / bottom edge belong to the next macro tile unless the image ends there
            const int jj = lane / 5, i = lane - jj * 5;
            const int gx = cx0 + i, gy = cy0 + jj;
            if (gx < C.latW && gy < C.latH) {
                const uint32_t tv = touch[lane];
                if (tv) atomicOr(&C.touchMap[(size_t)gy * C.latW + gx], tv);
                if ((i < 4 || wIn <= 16) && (jj < 4 || hIn <= 16)) {
                    uint8_t* d = C.latRGB + ((size_t)gy * C.latW + gx) * 3;
#pragma unroll
                    for (int c = 0; c < 3; c++) d[c] = (uint8_t)yk_compress250(yk_round6(priv[c * YKP_CH + (4 * jj) * YKP_RS + 4 * i]));
                }
            }
        }
    }
    if (threadIdx.x == 32) YKT(12);
    if (run.doR2 && claimed != 0xFFFFu) {
        const int tilesW = C.w >> 3;
#if YKA_RANGE_SINGLE
#pragma unroll 1
        for (int t8 = 0; t8 < 4; t8++) {
            const int qx = t8 & 1, qy = t8 >> 1;
            const unsigned c4 = claimed >> (8 * qy + 2 * qx);
            const unsigned q = (~((c4 & 3u) | (((c4 >> 4) & 3u) << 2))) & 15u;
            if (q) {
                const size_t tile = (size_t)((gmy + 8 * qy) >> 3) * tilesW + ((gmx + 8 * qx) >> 3);
                yka_range_tile(priv, C, hist, magicTab, tile, 8 * qx, 8 * qy, q);
            }
        }
#else
#pragma unroll 1
        for (int qy = 0; qy < 2; qy++) {
            // unclaimed cells of the two cell rows of this half, as quadrant masks of its left and right 8x8 tile
            const unsigned f = ~(claimed >> (8 * qy));
            const unsigned qL = (f & 3u) | ((f >> 2) & 12u), qR = ((f >> 2) & 3u) | ((f >> 4) & 12u);
            if (qL | qR) {
                const size_t tileL = (size_t)((gmy + 8 * qy) >> 3) * tilesW + (gmx >> 3);
                yka_range_pair(priv, C, hist, magicTab, tileL, 8 * qy, qL, qR);
            }
        }
#endif
    }
    if (threadIdx.x == 32) YKT(13);
}


template <bool U8>
static __device__ __forceinline__ void yk_analyze_body(const YkSlotDev* __restrict__ slots, int slot0, int nSlots, int nRegions, const YkRun& runArg) {
    // one dynamic shared-memory block, carved by constant offsets from the array itself so that every access stays in
    // the shared address space (LDS / STS / ATOMS, no generic loads)
#ifdef YK_EMULATE
    static __align__(128) unsigned char smem[YKA_SMEM_BYTES];
#else
    extern __shared__ __align__(128) unsigned char smem[];
#endif
    unsigned char* raw = smem;
    constexpr int STAGE_BYTES = U8 ? YKA_RAWB_STAGE : YKA_RAW_STAGE_INTS * 4;
    constexpr int PLANE_BYTES = U8 ? YKA_RAWB_PLANE : YKA_RAW_PLANE_INTS * 4;
    YkaWarpArea* warpAreas = reinterpret_cast<YkaWarpArea*>(smem + YKA_SMEM_RAW);
    uint32_t* sMagic = reinterpret_cast<uint32_t*>(smem + YKA_SMEM_RAW + YKA_SMEM_WARPS);    // ceil(2^20 / d): exact floor(n / d) for n < 4112, d <= 255
    YkaShared& sh = *reinterpret_cast<YkaShared*>(smem + YKA_SMEM_RAW + YKA_SMEM_WARPS + 1024);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef YK_TIMING
    if (tid == 0) { const unsigned long long n = ykt_now(); atomicMax(&yk_timing[30], ~n); atomicAdd(&yk_timing[31], n & 0xFFFFFFFFull); }
#endif
    // units of one image: (pair of regions, macro-tile row); every image of a launch has the same size
    const int nbxAll = slots[slot0].nbx, nPairs = (nbxAll + 1) >> 1;
    const int unitsPerSlot = nPairs * (nRegions / nbxAll) * 4, total = nSlots * unitsPerSlot;

    // the producer warp asks for what its first unit needs from global memory before the set-up below (the round trips
    // overlap the set-up instead of following it)
    const int firstSlot = slot0 + (YKA_STATIC_FIRST && nSlots > 1 ? (int)blockIdx.x / unitsPerSlot : 0);
    int firstPlanes = 0;
    int* ticket = nullptr;
    if (warp == 0) {
        firstPlanes = slots[firstSlot].nPlanes;
        ticket = slots[slot0].hdr + YK_HD_TICKET_ANALYZE;
        if (lane < 4) yka_tmap_acquire(&slots[firstSlot].tmap[lane]);        // all four: nothing here waits for a load
    }
    uint4 laneEntry = make_uint4(0u, 0u, 0u, 0u);
    if (tid >= 128 && tid < 128 + YK_NPASS * 32) laneEntry = *reinterpret_cast<const uint4*>(&yka_lane_table.e[(tid - 128) >> 5][(tid - 128) & 31]);
    // ---- start-up (the only block-wide barrier).  Nothing is cleared wholesale: every field that is read before it is
    // written has one thread that initialises it, and a consumer warp prepares its own area.
#if YKA_RANGE_SINGLE
    if (tid < 256) sMagic[tid] = tid ? ((1u << 20) + (unsigned)tid - 1u) / (unsigned)tid : 0u;
#else
    if (tid < 256) sMagic[tid] = tid ? (((1u << 22) + (unsigned)tid - 1u) / (unsigned)tid) << 9 : 0x80000000u;      // see yka_range_pair
#endif
    if (tid >= 384 && tid < 384 + YKA_NSTAT) sh.stat[tid - 384] = 0;
    if (warp >= 1) {
        YkaWarpArea& mine = warpAreas[warp - 1];
        for (int i = lane; i < (int)sizeof(mine.hist) / 16; i += 32) reinterpret_cast<uint4*>(mine.hist)[i] = make_uint4(0u, 0u, 0u, 0u);
        for (int i = lane; i < 40; i += 32) mine.wstat[i] = 0;
        if (lane < 28) mine.touch[lane] = 0u;
        if (lane == 0) mine.slotc.slot = -1;
    }
#ifdef YK_TIMING
    if (tid == 0) { const unsigned long long n = ykt_now(); atomicMax(&yk_timing[16], ~n); atomicAdd(&yk_timing[17], n & 0xFFFFFFFFull); atomicAdd(&yk_timing[23], 1ull); }
#endif
    if (tid < 41) sh.pretestTab[tid] = yka_pretest_entry(tid);
    if (tid >= 128 && tid < 128 + YK_NPASS * 32) sh.passLane[(tid - 128) >> 5][(tid - 128) & 31] = laneEntry;
    if (tid < 41) sh.passOfTile[tid] = (uint8_t)((tid >= 1) + (tid >= 3) + (tid >= 5) + (tid >= 9) + (tid >= 17) + (tid >= 25));
    if (warp == 3) {
        // the run's parameters, the tiles its passes cover (one lane per pass) and the barriers of the raw ring (one lane each):
        // every other warp waits for this at the barrier below, so it is spread over the lanes
        if (lane == 0) { sh.run = runArg; sh.queueHead = 0; sh.endSeq = INT_MAX; sh.statSlot = -1; sh.consLeft = YKA_CONS_WARPS; }
        __syncwarp();                                       // passId is read from the shared copy: indexing the kernel parameter by lane would put it on the stack
        unsigned rtLo = 0, rtHi = 0;
        if (lane < runArg.nPasses) {
            const int pid = sh.run.passId[lane];
            const YkGeomS g = yk_geom_s(pid);
            const unsigned long long rt = ((1ull << (256 >> (g.shx + g.shy))) - 1ull) << g.start;
            rtLo = (unsigned)rt; rtHi = (unsigned)(rt >> 32);
            sh.rpOf[pid] = lane;
        }
        rtLo = __reduce_or_sync(YK_FULL, rtLo); rtHi = __reduce_or_sync(YK_FULL, rtHi);
        if (lane == 0) sh.runTiles = ((unsigned long long)rtHi << 32) | rtLo;
        if (lane < YKA_NR) {
            yka_mbar_init(&sh.rawFull[lane], 1); yka_mbar_init(&sh.rawFree[lane], YKA_ITEMS); sh.unit[lane].seq = -1;
#ifndef YK_EMULATE
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
        }
    }
    __syncthreads();
    const YkRun& run = sh.run;

    if (warp == 0) {
        // ================================================== producer (warp 0: the oldest warp of its scheduler) ==================================================
        // u-th unit of this CTA -> raw buffer u % YKA_NR
        const bool wantAlpha = run.doAlpha != 0;
        // tickets: lane 0 holds YKA_TICKETS tickets in separate registers (the loop is unrolled by that many units), each
        // fetched YKA_TICKETS units ahead, so that the latency of the global atomic is never on the path of a unit.
        // Towards the end of the launch (fewer than `endgame` units left) tickets are taken only when they are needed and
        // the look-ahead shrinks to one unit, so that the last units go to whichever CTA is free.
        const int endgame = total - run.endgameUnits * (int)gridDim.x;
        bool lazy = false;
        int tk[YKA_TICKETS];
        // of the image the current unit belongs to (kept in registers while the slot does not change)
        int curSlot = -1, alpha = 0;
        const YkSlotDev* S = nullptr;
        // pair index -> (pair column, by) by a multiply-high (exact for index * nPairs < 2^32)
        const unsigned pairMagic = nPairs > 1 ? 0xFFFFFFFFu / (unsigned)nPairs + 1u : 0u;
        // tk[] holds ticket values as the counter returned them; unit = value + tbase.  YKA_TK_LAZY: to be taken when the unit comes up.
        constexpr int YKA_TK_LAZY = INT_MIN;
#if YKA_STATIC_FIRST
        // A CTA's first unit(s) are known without asking: unit r * grid + its own index, r < nStatic (one round of the
        // ticket registers when the launch is long enough, else one unit) - nothing to wait for before their loads are
        // issued.  The counter hands out the units after those; the first round of real tickets is taken with one atomic
        // once the static units' loads are on their way.
        const int nStatic = total >= YKA_STATIC_ROUND_MIN * (int)gridDim.x ? YKA_TICKETS : 1;
        const int tbase = nStatic * (int)gridDim.x;
#pragma unroll
        for (int r = 0; r < YKA_TICKETS; r++) tk[r] = (int)blockIdx.x + (r < nStatic ? r : 0) * (int)gridDim.x - tbase;
        // the image of the first unit (descriptors acquired at the top of the kernel)
        S = &slots[firstSlot];
        alpha = wantAlpha && firstPlanes == 4;
        curSlot = firstSlot;
        if (lane == 0) sh.statSlot = firstSlot;
#else
        const int nStatic = 0, tbase = 0;
#pragma unroll
        for (int r = 0; r < YKA_TICKETS; r++) { tk[r] = 0; if (lane == 0) tk[r] = atomicAdd(ticket, 1); }
#endif
        YKT_DECL;
#if YKA_PRODUCER_ROLLED
        static_assert(YKA_TICKETS == 4, "the rolled producer loop rotates four ticket registers");
#pragma unroll 1
        for (int u = 0;; u++) {
            {
                constexpr int r = 0;                         // the current unit's ticket is always in tk[0]: the registers rotate at the end of the body
                const int i = u % YKA_NR;
#else
        for (int u0 = 0;; u0 += YKA_TICKETS) {
#pragma unroll
            for (int r = 0; r < YKA_TICKETS; r++) {
                const int u = u0 + r, i = u % YKA_NR;
#endif
                // never more than YKA_LOOKAHEAD units ahead of the consumers: the CTAs then run out of work together
                while (u - (yka_flag_ld(&sh.queueHead) >> 3) > (lazy ? YKA_LAZY_AHEAD : YKA_LOOKAHEAD)) yk_spin();
                if (u >= YKA_NR) yka_mbar_wait(&sh.rawFree[i], (unsigned)((u / YKA_NR - 1) & 1));
                if (lane == 0) YKT(0);
                if (lane == 0 && tk[r] == YKA_TK_LAZY) tk[r] = atomicAdd(ticket, 1);           // endgame: taken on demand
                const int item = __shfl_sync(YK_FULL, tk[r], 0) + tbase;
                if (lane == 0) YKT(6);
                if (item >= total) { if (lane == 0) yka_flag_st(&sh.endSeq, u); return; }
                lazy = item >= endgame;
                int slot = slot0, rem = item;
                if (nSlots > 1) { const int q = item / unitsPerSlot; slot += q; rem -= q * unitsPerSlot; }
                if (slot != curSlot) {
                    S = &slots[slot];
                    if (lane < S->nPlanes) yka_tmap_acquire(&S->tmap[lane]);
                    alpha = wantAlpha && S->nPlanes == 4;
                    curSlot = slot;
                    if (u == 0 && lane == 0) sh.statSlot = slot;
                }
                const int pr = rem >> 2, k = rem & 3;
                const int by = nPairs > 1 ? (int)__umulhi((unsigned)pr, pairMagic) : pr, bx = 2 * (pr - by * nPairs);
                if (lane == 0) {
                    YKT(3);
                    YkaUnit& U = sh.unit[i];
                    U.slot = slot; U.bx = bx; U.by = by; U.k = k; U.alpha = alpha; U.seq = u;
                    unsigned char* dst = raw + i * STAGE_BYTES;
#ifndef YKA_NO_PROXY_FENCE
                    yka_fence_async();
#endif
                    yka_mbar_expect_tx(&sh.rawFull[i], (U8 ? YKA_COLORB_TX : YKA_COLOR_TX) + (alpha ? (U8 ? YKA_ALPHAB_TX : YKA_ALPHA_TX) : 0u));
                    for (int c = 0; c < 3; c++)
                        yka_tma_box(dst + c * PLANE_BYTES, &S->tmap[c], bx * 64, by * 64 + 16 * k, U8 ? YK_U8_BOX : YK_RAW_PITCH, YK_RAW_ROWS, &sh.rawFull[i], !alpha && c == 2);
                    if (alpha) yka_tma_box(dst + 3 * PLANE_BYTES, &S->tmap[3], bx * 64, by * 64 + 16 * k, YK_UNIT_W, 16, &sh.rawFull[i], 1);
                    YKT(2);
#ifdef YK_TIMING
                    if (u < 3) atomicAdd(&yk_timing[24 + u], ykt_now() & 0xFFFFFFFFull);
#endif
                    // the ticket this register holds next (used YKA_TICKETS units from now).  After the loads: the compiler
                    // turns an atomic on a uniform address into "leader adds, SHFL broadcasts" - inline PTX, atom.inc and a
                    // non-constant increment included - and that shuffle waits for the round trip to L2 where it stands.
                    if (u >= nStatic) tk[r] = lazy ? YKA_TK_LAZY : atomicAdd(ticket, 1);
                    else if (u == nStatic - 1) {
                        const int base = atomicAdd(ticket, YKA_TICKETS);
#pragma unroll
                        for (int j = 0; j < YKA_TICKETS; j++) tk[(r + 1 + j) % YKA_TICKETS] = base + j;      // units u + 1 .. u + YKA_TICKETS
                    }
                    YKT(7);
                }
#if YKA_PRODUCER_ROLLED
                { const int t0 = tk[0]; tk[0] = tk[1]; tk[1] = tk[2]; tk[2] = tk[3]; tk[3] = t0; }     // what was just taken is used four units from now
#endif
            }
        }
        return;
    }

    // ===================================================== consumers =====================================================
    const int cw = warp - 1;                                 // consumer index
    YkaWarpArea& WA = warpAreas[cw];
    uint8_t* hist = WA.hist;
    uint8_t* priv = WA.priv;
    uint32_t* touch = WA.touch;
    YkaSlotC& C = WA.slotc;
    YkaStat* st = WA.wstat;
    YKT_DECL;
    const bool fast16 = run.fresh && run.nPasses > 0 && run.passId[0] == 0;      // uniform for the launch
#ifdef YK_TIMING
    bool firstItem = true;
#endif
    for (;;) {
#ifdef YK_TIMING
        const long long tw0 = clock64();
#endif
        int q = 0;
        if (lane == 0) q = atomicAdd(&sh.queueHead, 1);
        q = __shfl_sync(YK_FULL, q, 0);
        const int u = q >> 3, mx = q & 7, i = u % YKA_NR;
        bool alive = true;
        // the unit of this item has been issued into raw buffer i (so the barrier's current phase is this unit's) and has
        // landed; the second wait suspends the warp.  Both look now and then whether the CTA has run out of units.
        while (yka_flag_ld(&sh.unit[i].seq) != u) {
            if (yka_flag_ld(&sh.endSeq) <= u) { alive = false; break; }
            yk_spin();
        }
        while (alive && !yka_mbar_try_wait(&sh.rawFull[i], (unsigned)((u / YKA_NR) & 1))) {
            if (yka_flag_ld(&sh.endSeq) <= u) { alive = false; break; }
        }
        alive = __all_sync(YK_FULL, alive);
        if (tid == 32) YKT(8);
#ifdef YK_TIMING
        if (lane == 0) { const unsigned long long dt = (unsigned long long)(clock64() - tw0); atomicAdd(&yk_timing[!alive ? 15 : firstItem ? 14 : 5], dt); if (alive && !firstItem) atomicAdd(&yk_timing[4], 1ull); }
        if (lane == 0 && firstItem && alive) { atomicAdd(&yk_timing[18], ykt_now() & 0xFFFFFFFFull); atomicAdd(&yk_timing[19], 1ull); if (u < 3 && mx == 0) atomicAdd(&yk_timing[27 + u], ykt_now() & 0xFFFFFFFFull); }
        firstItem = false;
#endif
        if (!alive) break;
        const YkaUnit U = sh.unit[i];
        const int cachedSlot = C.slot;
        __syncwarp();                                       // every lane has read the cached id before lane 0 may rewrite it
        if (cachedSlot != U.slot) {
            if (cachedSlot >= 0) yka_stat_flush(sh, C, st);     // the counters so far belong to the previous image
            yka_slot_refresh(slots[U.slot], C, U.slot);
        }
        const int X0 = U.bx * 64, Yk = U.by * 64 + 16 * U.k;
        const int gmx = X0 + 16 * mx;
        const unsigned char* rawU = raw + i * STAGE_BYTES;
#ifdef YKA_DEBUG_SKIP_WORK      // measurement only: how long the launch takes when the consumers only hand the raw rows back
        __syncwarp();
        if (lane == 0) yka_mbar_arrive(&sh.rawFree[i]);
        continue;
#endif
        // fresh state, 16x16 pass first, interior macro tile: try that pass straight from the raw rows
        int fast = 0;
        if (fast16 && gmx + 20 <= C.w && Yk + YK_RAW_ROWS <= C.h)
            fast = yka_pass16_raw<U8>(rawU, C, st, gmx, Yk, mx, run.rejectFactor);
        bool kept;
        if (fast == 1) {
            // accepted: the macro tile is finished without a byte tile; alpha test and the corner colours of its 4x4
            // lattice points (EC.cpp:4115-4132) come from the raw rows
            kept = U.alpha ? yka_alpha_any<U8>(rawU, mx) : false;
            if (lane < 16) {
                const int li = lane & 3, lj = lane >> 2;
                uint8_t* d = C.latRGB + ((size_t)((Yk >> 2) + lj) * C.latW + (gmx >> 2) + li) * 3;
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    const int v = U8 ? (int)rawU[c * YKA_RAWB_PLANE + 4 * lj * YK_U8_BOX + 16 * mx + 4 * li]
                                     : reinterpret_cast<const int32_t*>(rawU)[c * YKA_RAW_PLANE_INTS + 4 * lj * YK_RAW_PITCH + 16 * mx + 4 * li];
                    d[c] = (uint8_t)yk_compress250(yk_round6(v & 255));
                }
            }
        } else {
            kept = yka_pack_macro_tile<U8>(rawU, priv, C, X0, Yk, mx, U.alpha != 0);
        }
        __syncwarp();
        if (lane == 0) yka_mbar_arrive(&sh.rawFree[i]);      // this warp is done with the raw rows
        if (tid == 32) YKT(9);
        if (gmx >= C.w) continue;                            // the unit's second region does not exist (odd number of region columns)
        if (U.alpha && Yk < C.h) {
            if (lane == 0) C.alphaKept[(size_t)(Yk >> 4) * ((C.w + 15) >> 4) + (gmx >> 4)] = kept ? 1 : 0;
            // bounding box of kept tiles (EC.cpp:416-422), mins stored as extent - value so that zero means "none"
            if (kept) yka_stat_add(st, 7, 1, C.w - gmx, INT_MAX / 2 - (C.yOrg + Yk), min(gmx + 16, C.w), C.yOrg + min(Yk + 16, C.h));
        }
        if (fast == 1) continue;
        yka_macro_tile(priv, sh, C, touch, hist, sMagic, st, gmx, Yk, fast == 2);
        __syncwarp();
        if (tid == 32) YKT(10);
    }
#ifdef YK_TIMING
    if (lane == 0) { const unsigned long long n = ykt_now(); atomicAdd(&yk_timing[20], n & 0xFFFFFFFFull); atomicAdd(&yk_timing[21], 1ull); atomicMax(&yk_timing[22], n); }
#endif
    if (C.slot >= 0) yka_stat_flush(sh, C, st);
    // the last consumer warp of the CTA adds the CTA's counters to the image's header
    __threadfence_block();
    int left = 0;
    if (lane == 0) left = atomicSub(&sh.consLeft, 1);
    left = __shfl_sync(YK_FULL, left, 0);
    if (left == 1 && sh.statSlot >= 0) {
        __threadfence_block();
        int* hdr = slots[sh.statSlot].hdr;
        for (int idx = YK_HD_ALPHA_KEPT0 + lane; idx < YK_HD_INTS; idx += 32) {
            const int v = sh.stat[idx];
            if (v) {
                const int f = idx < YK_HD_PASS0 ? idx - YK_HD_ALPHA_KEPT0 : (idx - YK_HD_PASS0) % YK_ST_STRIDE;
                if (f == 0) atomicAdd(&hdr[idx], v); else atomicMax(&hdr[idx], v);
            }
        }
    }
}

__global__ void __launch_bounds__(YKA_THREADS, 1)
yk_k_analyze(const YkSlotDev* __restrict__ slots, int slot0, int nSlots, int nRegions, YkRun run) {
    yk_analyze_body<false>(slots, slot0, nSlots, nRegions, run);
}
// the same over planes uploaded packed to bytes by yk_set_image (a quarter of the HBM and PCIe traffic)
__global__ void __launch_bounds__(YKA_THREADS, 1)
yk_k_analyze_u8(const YkSlotDev* __restrict__ slots, int slot0, int nSlots, int nRegions, YkRun run) {
    yk_analyze_body<true>(slots, slot0, nSlots, nRegions, run);
}

// packed planes -> int32 planes, for the kernels outside the hot path that read Plane-style samples
__global__ void __launch_bounds__(256)
yk_k_expand(const YkSlotDev* __restrict__ slots, int slot, int w, int h, int32_t* d0, int32_t* d1, int32_t* d2, int32_t* d3) {
    const YkSlotDev& S = slots[slot];
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w || y >= h) return;
    int32_t* d[4] = { d0, d1, d2, d3 };
    for (int p = 0; p < S.nPlanes; p++) if (d[p]) d[p][(size_t)y * w + x] = S.planeU8[p][(size_t)y * S.pitchU8 + x];
}

// Interleaved 8-bit pixels (C = 3: R,G,B; 4: R,G,B,A; rows rowBytes apart) -> the slot's packed planes (yk_set_image_interleaved).
// A thread takes 16 pixels of a row: C uint4 loads when the rows are 16-byte aligned and all 16 pixels exist, else byte loads
// of the 4-pixel units inside the row (w is a multiple of 4), so that nothing past a row's last pixel is read.  One uint4
// store per plane; the packed row's padding gets zeros, as the host packing writes.
template <int C> static __device__ __forceinline__ uint32_t yk_unpack_unit(const uint32_t* u, int p) {
    // C words hold 4 pixels; byte C * i + p is sample p of pixel i
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) r |= ((u[(C * i + p) >> 2] >> (8 * ((C * i + p) & 3))) & 255u) << (8 * i);
    return r;
}
template <int C>
__global__ void __launch_bounds__(256)
yk_k_unpack8(YkUnpackArgs a) {
    const int groups = (a.w + 15) >> 4;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)groups * a.h) return;
    const int y = (int)(idx / groups), x0 = (int)(idx - (long long)y * groups) * 16;
    const uint8_t* row = a.src + (size_t)y * a.rowBytes + (size_t)x0 * C;
    uint32_t u[4 * C];
    if (((((uintptr_t)a.src) | a.rowBytes) & 15) == 0 && x0 + 16 <= a.w) {
#pragma unroll
        for (int k = 0; k < C; k++) {
            const uint4 v = reinterpret_cast<const uint4*>(row)[k];
            u[4 * k] = v.x; u[4 * k + 1] = v.y; u[4 * k + 2] = v.z; u[4 * k + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4 * C; k++) u[k] = 0;
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (x0 + 4 * j < a.w)
#pragma unroll
                for (int b = 0; b < 4 * C; b++) u[C * j + (b >> 2)] |= (uint32_t)row[4 * C * j + b] << (8 * (b & 3));
    }
    const size_t o = (size_t)y * a.pitch + x0;
#pragma unroll
    for (int p = 0; p < C; p++)
        if (p < a.nPlanes)
            *reinterpret_cast<uint4*>(a.dst[p] + o) = make_uint4(yk_unpack_unit<C>(u, p), yk_unpack_unit<C>(u + C, p),
                                                                 yk_unpack_unit<C>(u + 2 * C, p), yk_unpack_unit<C>(u + 3 * C, p));
}

// A new launch on a state that already holds claims: every touched lattice point becomes "claimed before" (bit 31).
__global__ void __launch_bounds__(256)
yk_k_fold_touch(const YkSlotDev* __restrict__ slots, int slot0, int nWords) {
    const YkSlotDev& S = slots[slot0 + blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nWords) { uint32_t v = S.touchMap[i]; if (v && v != 0x80000000u) S.touchMap[i] = 0x80000000u; }
}

// ------------------------------------------------------------------------------------------------------------------
int yk_analyze_setup(int* numSMs) {
#ifdef YK_EMULATE
    if (numSMs) *numSMs = 2;
    return 0;
#else
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    int n = 0;
    e = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return (int)e;
    if (numSMs) *numSMs = n;
    e = cudaFuncSetAttribute(yk_k_analyze, cudaFuncAttributeMaxDynamicSharedMemorySize, YKA_SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaFuncSetAttribute(yk_k_analyze_u8, cudaFuncAttributeMaxDynamicSharedMemorySize, YKA_SMEM_BYTES);
#endif
}
void yk_launch_analyze(const YkSlotDev* slotsDev, int slot0, int nSlots, int nRegions, int gridCtas, bool packedU8, const YkRun& run, cudaStream_t st) {
    const int total = nSlots * nRegions * 4;                 // units: macro-tile rows of regions
    const int grid = gridCtas < total ? gridCtas : total;
    if (packedU8) YK_LAUNCH(yk_k_analyze_u8, dim3(grid), dim3(YKA_THREADS), YKA_SMEM_BYTES, st, slotsDev, slot0, nSlots, nRegions, run);
    else YK_LAUNCH(yk_k_analyze, dim3(grid), dim3(YKA_THREADS), YKA_SMEM_BYTES, st, slotsDev, slot0, nSlots, nRegions, run);
}
void yk_launch_expand(const YkSlotDev* slotsDev, int slot, int nPlanes, int w, int h, int32_t* const* dst, cudaStream_t st) {
    YK_LAUNCH(yk_k_expand, dim3((w + 255) / 256, h), dim3(256), 0, st, slotsDev, slot, w, h, dst[0], dst[1], dst[2], nPlanes > 3 ? dst[3] : (int32_t*)nullptr);
}
void yk_launch_unpack8(const YkUnpackArgs& a, int channels, cudaStream_t st) {
    const long long threads = (long long)((a.w + 15) >> 4) * a.h;
    const dim3 grid((unsigned)((threads + 255) / 256));
    if (channels == 4) YK_LAUNCH(yk_k_unpack8<4>, grid, dim3(256), 0, st, a);
    else YK_LAUNCH(yk_k_unpack8<3>, grid, dim3(256), 0, st, a);
}
void yk_launch_fold_touch(const YkSlotDev* slotsDev, int slot0, int nSlots, int nWords, cudaStream_t st) {
    YK_LAUNCH(yk_k_fold_touch, dim3((nWords + 255) / 256, nSlots), dim3(256), 0, st, slotsDev, slot0, nWords);
}

// CUDA loads kernels lazily, and loading one synchronises the context: a kernel that waits for another stream (yk_strip_run)
// would then never be released by a kernel that is launched for the first time.  Every kernel is loaded up front.
int yk_preload_analyze() {
#ifndef YK_EMULATE
    cudaFuncAttributes fa;
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_analyze); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_analyze_u8); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_expand); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_unpack8<3>); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_unpack8<4>); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_fold_touch); if (e != cudaSuccess) return (int)e; }
#endif
    return 0;
}
