// Device-side helpers shared by the kernel translation units (yk_analyze.cu, yk_emit.cu, yk_kernels.cu).
// Reference line numbers are KLab/YAIK's encoder/EncoderContext.cpp ("EC.cpp") unless another file is named.
#pragma once
#include "yk_internal.h"
#include <limits.h>

#define YK_RS 72                 // shared-memory row pitch in bytes of a staged 65x65 byte tile (18 words: conflict-free rows)
#define YK_PIXTILE (65 * YK_RS)  // bytes of one staged channel
#define YK_FULL 0xffffffffu

static __device__ __forceinline__ int yk_round6(int v) { int r = v >> 2; return (r << 2) | (r >> 4); }                 // EC.cpp:3183-3189
static __device__ __forceinline__ int yk_round6p(int v) { v = min(v + 1, 255); int r = v >> 2; return (r << 2) | (r >> 4); }  // EC.cpp:3202-3207
static __device__ __forceinline__ int yk_compress250(int v) { return (v * 250 + 127) / 255; }                          // CompressF(v, colorCompressionQuad), EC.cpp:3191-3194

// Swizzle geometry with shifts (HeaderGradientTile::getSwizzleSize, include/YAIK_private.h:212-276), Convert()'s pass
// order (EC.cpp:9057-9093).  start = first bit of the pass inside the 41-bit "tiles of a macro tile" words.
struct YkGeomS { int shx, shy, lbw, lbh, bits, start; };
__constant__ YkGeomS yk_geom_s_tab[YK_NPASS] = { {4,4,6,6,16,0}, {4,3,6,6,32,1}, {3,4,6,6,32,3}, {3,3,6,6,64,5}, {3,2,6,5,64,9}, {2,3,5,6,64,17}, {2,2,5,5,64,25} };
static __device__ __forceinline__ YkGeomS yk_geom_s(int pid) { return yk_geom_s_tab[pid]; }

// stream position (== bitmap bit index) of the tile at global tile coords (gtx, gty), EC.cpp:3801-3828, 4227-4234
static __device__ __forceinline__ int yk_pos_s(const YkGeomS& g, int nSwzX, int gtx, int gty) {
    const int x = gtx << g.shx, y = gty << g.shy;
    return (((y >> g.lbh) * nSwzX + (x >> g.lbw)) * g.bits) + (((y & ((1 << g.lbh) - 1)) >> g.shy) << (g.lbw - g.shx)) + ((x & ((1 << g.lbw) - 1)) >> g.shx);
}

// ------------------------------------------------------------------------------------------------------------------
// volatile access + decoupled look-back.  Work units are handed out by an atomic ticket in stream order, so a unit only
// ever waits for units with smaller tickets, which are already running or finished.
#ifdef YK_EMULATE
static inline unsigned yk_ldv(const unsigned* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline void yk_stv(unsigned* p, unsigned v) { __atomic_store_n(p, v, __ATOMIC_SEQ_CST); }
static inline int yk_ldvi(const int* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline void yk_stvi(int* p, int v) { __atomic_store_n(p, v, __ATOMIC_SEQ_CST); }
static inline unsigned long long yk_ldv64(const unsigned long long* p) { return __atomic_load_n(p, __ATOMIC_SEQ_CST); }
static inline void yk_stv64(unsigned long long* p, unsigned long long v) { __atomic_store_n(p, v, __ATOMIC_SEQ_CST); }
static inline void yk_spin() { std::this_thread::yield(); }
#else
static __device__ __forceinline__ unsigned yk_ldv(const unsigned* p) { return *reinterpret_cast<const volatile unsigned*>(p); }
static __device__ __forceinline__ void yk_stv(unsigned* p, unsigned v) { *reinterpret_cast<volatile unsigned*>(p) = v; }
static __device__ __forceinline__ int yk_ldvi(const int* p) { return *reinterpret_cast<const volatile int*>(p); }
static __device__ __forceinline__ void yk_stvi(int* p, int v) { *reinterpret_cast<volatile int*>(p) = v; }
static __device__ __forceinline__ unsigned long long yk_ldv64(const unsigned long long* p) { return *reinterpret_cast<const volatile unsigned long long*>(p); }
static __device__ __forceinline__ void yk_stv64(unsigned long long* p, unsigned long long v) { *reinterpret_cast<volatile unsigned long long*>(p) = v; }
static __device__ __forceinline__ void yk_spin() { __nanosleep(20); }
#endif

// status word: hi << 32 | lo << 2 | flag (1 = this unit's own totals, 2 = inclusive prefix).  Returns the exclusive prefix of
// unit u and publishes its inclusive prefix.  All 32 lanes call it with the same arguments.
static __device__ unsigned long long yk_lookback64(unsigned long long* status, int u, unsigned hi, unsigned lo) {
    const int lane = threadIdx.x & 31;
    const unsigned long long mine = ((unsigned long long)hi << 32) | ((unsigned long long)lo << 2);
    if (u == 0) { if (lane == 0) yk_stv64(&status[0], mine | 2ull); return 0ull; }
    if (lane == 0) yk_stv64(&status[u], mine | 1ull);
    unsigned bhi = 0, blo = 0;
    int look = u - 1;
    while (look >= 0) {
        const int idx = look - lane;
        const unsigned long long st = idx >= 0 ? yk_ldv64(&status[idx]) : 2ull;
        const unsigned fl = (unsigned)(st & 3ull);
        const unsigned ready = __ballot_sync(YK_FULL, fl != 0u);
        const unsigned incl = __ballot_sync(YK_FULL, fl == 2u);
        const unsigned need = incl ? ((2u << (__ffs((int)incl) - 1)) - 1u) : YK_FULL;
        if ((ready & need) != need) { yk_spin(); continue; }
        const bool use = (need >> lane) & 1u;
        bhi += __reduce_add_sync(YK_FULL, use ? (unsigned)(st >> 32) : 0u);
        blo += __reduce_add_sync(YK_FULL, use ? (unsigned)((st & 0xFFFFFFFFull) >> 2) : 0u);
        if (incl) break;
        look -= 32;
    }
    if (lane == 0) yk_stv64(&status[u], (((unsigned long long)(bhi + hi)) << 32) | ((unsigned long long)(blo + lo) << 2) | 2ull);
    return ((unsigned long long)bhi << 32) | blo;
}
