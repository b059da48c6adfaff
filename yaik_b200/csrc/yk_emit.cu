// yaik_b200 — corner ownership, rgbStream emission and the gather of the range stage's streams (sm_100a).
//
// The reference walks tiles in stream order and lets a tile emit a corner colour only if no earlier tile (of this or an
// earlier pass) touched that lattice point (mappedRGB, EC.cpp:4001-4021, 4115-4132).  Order-free: a lattice point is
// emitted in the first pass that touches it, by the accepted toucher with the smallest stream position — all of which
// the point's touch word says (written by yk_k_analyze).
//
//   yk_k_owner   one thread per lattice point: resolves the owner and sets the owner tile's bit in emitNib
//                (4 bits per tile in stream order: it emits TL / TR / BL / BR), and counts the group totals yk_k_emit
//                takes its offsets from: the point's 3 bytes for its owner tile's group, one range tile per even point.
//   yk_k_emit    one CTA per group of 8 x YK_EMIT_THREADS tiles of a pass: byte counts from the nibbles (popc), block scan,
//                the group's base = the totals of the groups before it in stream order, then the colours are copied from
//                latRGB.  CTAs past the gradient groups gather DynamicTileCompressor's per-tile output (written at fixed
//                places by yk_k_analyze) into the reference's row-major tile order (EC.cpp:8412-8413), offsets by the
//                same scan + base.
// Every total a base sums is final before yk_k_emit starts, so its CTAs run in any order and none waits for another.  The
// totals have two levels (groups, super-groups of YK_SUPER groups): a base costs at most YK_SUPER - 1 + G / YK_SUPER loads.
#include "yk_device.h"
#ifdef YK_EMULATE
#include <assert.h>
#endif

// Strips (one large image split into tile-row strips over several GPUs, SURVEY.md 8e): the lattice row on a strip
// boundary is touched by tiles of both strips.  Each strip ORs in the words its neighbour computed (touchInTop /
// touchInBottom); a tile of the upper strip always precedes a tile of the lower strip in a pass's stream, and only the
// strip that holds the owner tile marks it.
#ifndef YK_OWNER_THREADS
#define YK_OWNER_THREADS 256
#endif
// The owner of lattice point idx: sets its bit in emitNib and returns pass id << 24 | the owner tile's group, or -1 when
// this strip emits nothing there.
static __device__ __forceinline__ int yk_owner_point(const YkSlotDev& S, int idx, const YkRun& run) {
    uint32_t word = __ldg(&S.touchMap[idx]);
    const int gy = idx / S.latW, gx = idx - gy * S.latW;
    if (S.hasAbove && gy == 0) word |= __ldg(&S.touchInTop[gx]);
    if (S.hasBelow && gy == S.latH - 1) word |= __ldg(&S.touchInBottom[gx]);
    if (word == 0u || (word & 0x80000000u)) return -1;              // untouched / claimed by an earlier launch
    const int rp = (__ffs((int)(word & 0x0FFFFFFFu)) - 1) >> 2;     // first pass of this launch that touches the point
    const unsigned nib = (word >> (4 * rp)) & 15u;                  // roles present in that pass
    const int pid = run.passId[rp];
    const YkGeomS g = yk_geom_s(pid);
    const int nSwzX = (S.w + (1 << g.lbw) - 1) >> g.lbw;
    const int LX = (4 * gx) >> g.shx, LY = (4 * gy) >> g.shy;       // the point in tile units of that pass
    const int tileRows = S.h >> g.shy;
    int best = INT_MAX, bestK = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if ((nib >> k) & 1u) {                                      // an accepted tile has the point as its corner k
            const int ty = LY - (k >> 1);
            int pos;
            if (ty < 0) pos = k - 5;                                // a tile of the strip above: before every tile of this strip (BR's tile before BL's)
            else if (ty >= tileRows) pos = INT_MAX - 1;             // a tile of the strip below: after every tile of this strip
            else pos = yk_pos_s(g, nSwzX, LX - (k & 1), ty);
            if (pos < best) { best = pos; bestK = k; }
        }
    }
    if (best < 0 || best == INT_MAX - 1) return -1;                 // the neighbouring strip holds the owner
    atomicOr(&S.emitNib[pid][best >> 3], 1u << (4 * (best & 7) + bestK));
    return (pid << 24) | (int)((unsigned)(best >> 3) / YK_EMIT_THREADS);
}

static __device__ __forceinline__ void yk_rgb_add(const YkSlotDev& S, int key, unsigned bytes) {
    const unsigned grp = (unsigned)key & 0xFFFFFFu;
    atomicAdd(&S.rgbTot[key >> 24][grp], bytes);
    atomicAdd(&S.rgbSup[key >> 24][grp / YK_SUPER], bytes);
}
// sum: chunks << 16 | coded tiles (of at most one CTA of yk_k_owner: the fields do not overlap)
static __device__ __forceinline__ void yk_r2_add(const YkSlotDev& S, int grp, unsigned sum) {
    const unsigned long long v = (unsigned long long)(sum >> 16) << 32 | (sum & 0xFFFFu);
    atomicAdd(&S.r2Tot[grp], v);
    atomicAdd(&S.r2Sup[grp / YK_SUPER], v);
}

// R2: the coded quadrants of 8x8 tile (tx, ty), as chunks << 16 | 1 (0: not coded); the rule of yk_k_emit
static __device__ __forceinline__ unsigned yk_r2_count(const YkSlotDev& S, int tx, int ty) {
    const uint32_t r0 = S.cellMask[(size_t)(2 * ty) * S.nbx + (tx >> 3)], r1 = S.cellMask[(size_t)(2 * ty + 1) * S.nbx + (tx >> 3)];
    const int s2 = 2 * (tx & 7);
    const unsigned chunks = 4u - (unsigned)__popc(((r0 >> s2) & 3u) | (((r1 >> s2) & 3u) << 2));   // quadrants whose top-left map pixel is 0 (EC.cpp:8420-8430)
    return chunks ? chunks << 16 | 1u : 0u;
}

// The group totals yk_k_emit takes its bases from.  rgbStreams: 3 bytes per emitted lattice point, to its owner tile's group.
// R2 (run.doR2): the thread of lattice point (2 tx, 2 ty) counts tile (tx, ty), whose cells are final after the analysis.
// The points of a CTA (256 consecutive points of a lattice row) have their owner tiles, per pass, and their tiles nearly
// always in one group: a warp sums equal keys with one lane, the CTA sums each pass's largest key in shared memory and adds
// it once.  Adds from every warp to the same few words would queue at the L2.
__global__ void __launch_bounds__(YK_OWNER_THREADS)
yk_k_owner(const YkSlotDev* __restrict__ slots, int slot0, int nPoints, int owners, YkRun run) {
    __shared__ int sKey[YK_NPASS + 1];              // [YK_NPASS]: R2
    __shared__ unsigned sSum[YK_NPASS + 1];
    if (threadIdx.x <= YK_NPASS) { sKey[threadIdx.x] = -1; sSum[threadIdx.x] = 0u; }
    __syncthreads();
    const YkSlotDev& S = slots[slot0 + blockIdx.y];
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int key = owners && idx < nPoints ? yk_owner_point(S, idx, run) : -1;
    int r2Key = -1;
    unsigned r2 = 0u;
    if (run.doR2 && idx < nPoints) {
        const int gy = idx / S.latW, gx = idx - gy * S.latW, tx = gx >> 1, ty = gy >> 1;
        if (!((gx | gy) & 1) && tx < (S.w >> 3) && ty < (S.h >> 3)) {
            r2 = yk_r2_count(S, tx, ty);
            if (r2) r2Key = (int)((unsigned)(ty * (S.w >> 3) + tx) / YK_EMIT_THREADS);
        }
    }
    // a warp whose keys agree adds with one lane
    const unsigned rgbLanes = __ballot_sync(YK_FULL, key >= 0), r2Lanes = __ballot_sync(YK_FULL, r2Key >= 0);
    const int rgbTop = __reduce_max_sync(YK_FULL, key), r2Top = __reduce_max_sync(YK_FULL, r2Key);
    const bool rgbOne = __all_sync(YK_FULL, key < 0 || key == rgbTop), r2One = __all_sync(YK_FULL, r2Key < 0 || r2Key == r2Top);
    const unsigned r2Warp = __reduce_add_sync(YK_FULL, r2);
    const bool addRgb = key >= 0 && (!rgbOne || lane == __ffs((int)rgbLanes) - 1);
    const bool addR2 = r2Key >= 0 && (!r2One || lane == __ffs((int)r2Lanes) - 1);
    const unsigned rgbBytes = rgbOne ? 3u * (unsigned)__popc(rgbLanes) : 3u, r2Sum = r2One ? r2Warp : r2;
    if (addRgb) atomicMax(&sKey[key >> 24], key);
    if (addR2) atomicMax(&sKey[YK_NPASS], r2Key);
    __syncthreads();
    if (addRgb) {
        if (sKey[key >> 24] == key) atomicAdd(&sSum[key >> 24], rgbBytes);
        else yk_rgb_add(S, key, rgbBytes);                          // another group of the same pass in this CTA
    }
    if (addR2) {
        if (sKey[YK_NPASS] == r2Key) atomicAdd(&sSum[YK_NPASS], r2Sum);
        else yk_r2_add(S, r2Key, r2Sum);
    }
    __syncthreads();
    if (threadIdx.x < YK_NPASS && sSum[threadIdx.x]) yk_rgb_add(S, sKey[threadIdx.x], sSum[threadIdx.x]);
    if (threadIdx.x == YK_NPASS && sSum[YK_NPASS]) yk_r2_add(S, sKey[YK_NPASS], sSum[YK_NPASS]);
}

// Block scan of the per-thread counts (c, d) plus the block sum of the per-thread base shares (pc, pd): returns the
// thread's exclusive offsets (base + scan), and the block's own totals in totC / totD (every thread).
static __device__ __forceinline__ void yk_emit_scan(unsigned c, unsigned d, unsigned pc, unsigned pd, unsigned& offC, unsigned& offD,
                                                    unsigned& totC, unsigned& totD) {
    constexpr int NW = YK_EMIT_THREADS / 32;
    __shared__ unsigned sC[NW], sD[NW], sPC[NW], sPD[NW], sTot[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned ic = c, id = d;
#pragma unroll
    for (int k = 1; k < 32; k <<= 1) {
        const unsigned a0 = __shfl_up_sync(YK_FULL, ic, k), a1 = __shfl_up_sync(YK_FULL, id, k);
        if (lane >= k) { ic += a0; id += a1; }
    }
    pc = __reduce_add_sync(YK_FULL, pc); pd = __reduce_add_sync(YK_FULL, pd);
    if (lane == 31) { sC[warp] = ic; sD[warp] = id; }
    if (lane == 0) { sPC[warp] = pc; sPD[warp] = pd; }
    __syncthreads();
    if (warp == 0) {
        const unsigned a = lane < NW ? sC[lane] : 0u, b = lane < NW ? sD[lane] : 0u;
        const unsigned bc = __reduce_add_sync(YK_FULL, lane < NW ? sPC[lane] : 0u), bd = __reduce_add_sync(YK_FULL, lane < NW ? sPD[lane] : 0u);
        unsigned ia = a, ib = b;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            const unsigned a0 = __shfl_up_sync(YK_FULL, ia, k), a1 = __shfl_up_sync(YK_FULL, ib, k);
            if (lane >= k) { ia += a0; ib += a1; }
        }
        if (lane < NW) { sC[lane] = bc + ia - a; sD[lane] = bd + ib - b; }
        if (lane == 31) { sTot[0] = ia; sTot[1] = ib; }
    }
    __syncthreads();
    offC = sC[warp] + ic - c; offD = sD[warp] + id - d;
    totC = sTot[0]; totD = sTot[1];
}

// 512 threads (32 registers): per pipelined step 41.2 us, 256 threads 41.3, 128 threads 42.3 (DESIGN.md §7, round-3 A/B log)
__global__ void __launch_bounds__(YK_EMIT_THREADS)
yk_k_emit(const YkSlotDev* __restrict__ slots, int slot0, YkRun run, int gradGroups, int r2Groups) {
    const YkSlotDev& S = slots[slot0 + blockIdx.y];
    const int tid = threadIdx.x;
    const int w = S.w, h = S.h;

    if ((int)blockIdx.x >= gradGroups) {
        // ---- DynamicTileCompressor streams: tiles in row-major order, 16 bytes per coded quadrant, 3 type bytes per coded tile
        const int grp = blockIdx.x - gradGroups, tilesW = w >> 3, nTiles = tilesW * (h >> 3);
        // this thread's share of the group's base: a group before it in its super-group, earlier super-groups
        unsigned long long pre = tid < grp % YK_SUPER ? S.r2Tot[grp - grp % YK_SUPER + tid] : 0ull;
        for (int s = tid; s < grp / YK_SUPER; s += YK_EMIT_THREADS) pre += S.r2Sup[s];
        const int t = grp * YK_EMIT_THREADS + tid;
        const unsigned c = t < nTiles ? yk_r2_count(S, t % tilesW, t / tilesW) : 0u;
        const unsigned chunks = c >> 16;
        const unsigned tiles = chunks > 0;
        unsigned chunkOff, tileOff, totC, totT;
        yk_emit_scan(chunks, tiles, (unsigned)(pre >> 32), (unsigned)pre, chunkOff, tileOff, totC, totT);
#ifdef YK_EMULATE
        if (tid == 0) assert(((unsigned long long)totC << 32 | totT) == S.r2Tot[grp]);     // yk_k_owner counted the same tiles
#endif
        if (grp == r2Groups - 1 && tid == 0) { S.hdr[YK_HD_R2_CHUNKS] = (int)(chunkOff + totC); S.hdr[YK_HD_R2_TILES] = (int)(tileOff + totT); }
        if (chunks) {
#pragma unroll 1
            for (int p = 0; p < 3; p++) {
                const uint4* src = reinterpret_cast<const uint4*>(S.r2Raw[p] + (size_t)t * 64);
                uint4* dst = reinterpret_cast<uint4*>(S.r2Idx[p] + (size_t)chunkOff * 16);
                for (int k = 0; k < (int)chunks; k++) dst[k] = src[k];
                const uint32_t ty = S.r2RawType[p][t];
                uint8_t* td = S.r2Type[p] + (size_t)tileOff * 3;                                // EC.cpp:8503-8505
                td[0] = (uint8_t)ty; td[1] = (uint8_t)(ty >> 8); td[2] = (uint8_t)(ty >> 16);
            }
        }
        return;
    }

    // ---- rgbStream of one pass: CTA -> (pass position, group of 8 x YK_EMIT_THREADS tiles)
    int rp = 0, grp = blockIdx.x, nWords = 0, nSwzX = 0, nGroups = 0;
    YkGeomS g = yk_geom_s(run.passId[0]);
    for (;;) {
        g = yk_geom_s(run.passId[rp]);
        nSwzX = (w + (1 << g.lbw) - 1) >> g.lbw;
        nWords = (nSwzX * ((h + (1 << g.lbh) - 1) >> g.lbh) * g.bits) >> 3;
        nGroups = (nWords + YK_EMIT_THREADS - 1) / YK_EMIT_THREADS;
        if (grp < nGroups) break;
        grp -= nGroups; rp++;
    }
    const int pid = run.passId[rp];
    unsigned pre = tid < grp % YK_SUPER ? S.rgbTot[pid][grp - grp % YK_SUPER + tid] : 0u;
    for (int s = tid; s < grp / YK_SUPER; s += YK_EMIT_THREADS) pre += S.rgbSup[pid][s];
    const int wi = grp * YK_EMIT_THREADS + tid;
    uint32_t word = wi < nWords ? __ldg(&S.emitNib[pid][wi]) : 0u;
    const unsigned cnt = 3u * (unsigned)__popc(word);
    unsigned off, tot, unused0, unused1;
    yk_emit_scan(cnt, 0u, pre, 0u, off, unused0, tot, unused1);
#ifdef YK_EMULATE
    if (tid == 0) assert(tot == S.rgbTot[pid][grp]);                                            // yk_k_owner counted the same corners
#endif
    if (grp == nGroups - 1 && tid == 0) S.hdr[YK_HD_PASS0 + pid * YK_ST_STRIDE + YK_ST_RGBBYTES] = (int)(off + tot);
    if (word == 0u) return;
    // the 8 tiles of a word share a swizzle block: invert the stream position once
    const int lbits = g.bits == 16 ? 4 : (g.bits == 32 ? 5 : 6);
    const int pos0 = wi * 8, blk = pos0 >> lbits, within0 = pos0 & (g.bits - 1);
    const int tprShift = g.lbw - g.shx;
    const int bys = blk / nSwzX, bxs = blk - bys * nSwzX;
    uint8_t* out = S.rgb[pid];
    while (word) {
        const int b = __ffs((int)word) - 1;
        word &= word - 1u;
        const int within = within0 + (b >> 2), k = b & 3;                         // TL, TR, BL, BR (EC.cpp:4115-4132)
        const int gtx = (bxs << tprShift) + (within & ((1 << tprShift) - 1)), gty = (bys << (g.lbh - g.shy)) + (within >> tprShift);
        const int gx = ((gtx + (k & 1)) << g.shx) >> 2, gy = ((gty + (k >> 1)) << g.shy) >> 2;
        const uint8_t* sp = S.latRGB + ((size_t)gy * S.latW + gx) * 3;
        out[off] = sp[0]; out[off + 1] = sp[1]; out[off + 2] = sp[2];
        off += 3;
    }
}

void yk_launch_owner(const YkSlotDev* slotsDev, int slot0, int nSlots, int nPoints, bool owners, const YkRun& run, cudaStream_t st) {
    YK_LAUNCH(yk_k_owner, dim3((nPoints + YK_OWNER_THREADS - 1) / YK_OWNER_THREADS, nSlots), dim3(YK_OWNER_THREADS), 0, st, slotsDev, slot0, nPoints, owners ? 1 : 0, run);
}
void yk_launch_emit(const YkSlotDev* slotsDev, int slot0, int nSlots, int gradGroups, int r2Groups, const YkRun& run, cudaStream_t st) {
    YK_LAUNCH(yk_k_emit, dim3(gradGroups + r2Groups, nSlots), dim3(YK_EMIT_THREADS), 0, st, slotsDev, slot0, run, gradGroups, r2Groups);
}

// Strips (yk_strip_run): epoch flags in halo memory.  The setter runs after the copies it announces (stream order) and
// makes them visible system-wide before the flag; the waiter spins on its own GPU's memory.
__global__ void yk_k_flag_set(unsigned* a, unsigned* b, unsigned value) {
    __threadfence_system();
    if (a) yk_stv(a, value);
    if (b) yk_stv(b, value);
}
__global__ void yk_k_flag_wait(const unsigned* a, const unsigned* b, unsigned value) {
    while (a && (int)(yk_ldv(a) - value) < 0) yk_spin();
    while (b && (int)(yk_ldv(b) - value) < 0) yk_spin();
    __threadfence_system();
}
void yk_launch_flag_set(unsigned* a, unsigned* b, unsigned value, cudaStream_t st) { YK_LAUNCH(yk_k_flag_set, dim3(1), dim3(1), 0, st, a, b, value); }
void yk_launch_flag_wait(const unsigned* a, const unsigned* b, unsigned value, cudaStream_t st) { YK_LAUNCH(yk_k_flag_wait, dim3(1), dim3(1), 0, st, a, b, value); }

// CUDA loads kernels lazily, and loading one synchronises the context: a kernel that waits for another stream (yk_strip_run)
// would then never be released by a kernel that is launched for the first time.  Every kernel is loaded up front.
int yk_preload_emit() {
#ifndef YK_EMULATE
    cudaFuncAttributes fa;
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_owner); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_emit); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_flag_set); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_flag_wait); if (e != cudaSuccess) return (int)e; }
#endif
    return 0;
}
