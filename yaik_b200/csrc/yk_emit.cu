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
//                the group's base = the totals of the groups before it in stream order, then the lattice points of the
//                group's corners are listed in shared memory and the whole CTA copies their colours from latRGB.  CTAs
//                past the gradient groups gather DynamicTileCompressor's per-tile output (written at fixed places by
//                yk_k_analyze) into the reference's row-major tile order (EC.cpp:8412-8413), offsets by the same scan +
//                base, the 16-byte chunks again from a list over the whole CTA.
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
#define YK_OWNER_THREADS 256
// The pass ids of a launch in run order, 4 bits each.  A kernel that indexed run.passId with a position known only at run
// time would copy the whole YkRun to local memory first.
static __device__ __forceinline__ unsigned yk_pass_ids(const YkRun& run) {
    unsigned v = 0u;
#pragma unroll
    for (int i = 0; i < YK_NPASS; i++) v |= ((unsigned)run.passId[i] & 15u) << (4 * i);
    return v;
}
static __device__ __forceinline__ int yk_pass_at(unsigned ids, int rp) { return (int)(ids >> (4 * rp)) & 15; }

// The owner of lattice point (gx, gy), whose touch word is non-zero and unclaimed: returns pass id << 24 | the owner tile's
// group and sets posK = the owner tile's stream position << 2 | its corner, or returns -1 when this strip emits nothing there.
static __device__ __forceinline__ int yk_owner_point(int w, int h, uint32_t word, int gx, int gy, unsigned passIds, int& posK) {
    const int rp = (__ffs((int)(word & 0x0FFFFFFFu)) - 1) >> 2;     // first pass of this launch that touches the point
    const unsigned nib = (word >> (4 * rp)) & 15u;                  // roles present in that pass
    const int pid = yk_pass_at(passIds, rp);
    const YkGeomS g = yk_geom_s(pid);
    const int nSwzX = (w + (1 << g.lbw) - 1) >> g.lbw;
    const int LX = (4 * gx) >> g.shx, LY = (4 * gy) >> g.shy;       // the point in tile units of that pass
    const int tileRows = h >> g.shy;
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
    posK = best << 2 | bestK;
    return (pid << 24) | (int)((unsigned)(best >> 3) / YK_EMIT_THREADS);
}

static __device__ __forceinline__ void yk_rgb_add(uint32_t* tot, uint32_t* sup, int key, unsigned bytes) {
    const unsigned grp = (unsigned)key & 0xFFFFFFu;
    atomicAdd(&tot[grp], bytes);
    atomicAdd(&sup[grp / YK_SUPER], bytes);
}
// sum: chunks << 16 | coded tiles (of at most one CTA of yk_k_owner: the fields do not overlap)
static __device__ __forceinline__ void yk_r2_add(unsigned long long* tot, unsigned long long* sup, int grp, unsigned sum) {
    const unsigned long long v = (unsigned long long)(sum >> 16) << 32 | (sum & 0xFFFFu);
    atomicAdd(&tot[grp], v);
    atomicAdd(&sup[grp / YK_SUPER], v);
}

// R2: the coded quadrants of 8x8 tile tx, as chunks << 16 | 1 (0: not coded), from the cellMask words of the tile's two
// cell rows; the rule of both kernels
static __device__ __forceinline__ unsigned yk_r2_rule(uint32_t r0, uint32_t r1, int tx) {
    const int s2 = 2 * (tx & 7);
    const unsigned chunks = 4u - (unsigned)__popc(((r0 >> s2) & 3u) | (((r1 >> s2) & 3u) << 2));   // quadrants whose top-left map pixel is 0 (EC.cpp:8420-8430)
    return chunks ? chunks << 16 | 1u : 0u;
}
static __device__ __forceinline__ unsigned yk_r2_count(const YkSlotDev& S, int tx, int ty) {
    const uint16_t* cm = S.cellMask + (size_t)(2 * ty) * S.nbx + (tx >> 3);
    return yk_r2_rule(cm[0], cm[S.nbx], tx);
}

// The group totals yk_k_emit takes its bases from.  rgbStreams: 3 bytes per emitted lattice point, to its owner tile's group.
// R2 (run.doR2): the thread of lattice point (2 tx, 2 ty) counts tile (tx, ty), whose cells are final after the analysis.
// The points of a CTA (256 consecutive points of a lattice row) have their owner tiles, per pass, and their tiles nearly
// always in one group: a warp sums equal keys with one lane, the CTA sums each pass's largest key in shared memory and adds
// it once.  Adds from every warp to the same few words would queue at the L2.
// Every load is issued ahead of the first atomic, the cellMask words beside the touch words: the compiler orders no load
// after an atomic, so nothing is reloaded behind the atomicOr and the R2 count adds no chain of its own.
__global__ void __launch_bounds__(YK_OWNER_THREADS)
yk_k_owner(const YkSlotDev* __restrict__ slots, int slot0, int nPoints, int owners, YkRun run) {
    __shared__ int sKey[YK_NPASS + 1];              // [YK_NPASS]: R2
    __shared__ unsigned sSum[YK_NPASS + 1];
    if (threadIdx.x <= YK_NPASS) { sKey[threadIdx.x] = -1; sSum[threadIdx.x] = 0u; }
    const YkSlotDev& S = slots[slot0 + blockIdx.y];
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int w = S.w, h = S.h, latW = S.latW, gy = idx / latW, gx = idx - gy * latW;
    const bool r2Point = run.doR2 && idx < nPoints && !((gx | gy) & 1) && (gx >> 1) < (w >> 3) && (gy >> 1) < (h >> 3);
    uint32_t word = 0u, m0 = 0u, m1 = 0u;
    if (owners && idx < nPoints) {
        word = __ldg(&S.touchMap[idx]);
        if (S.hasAbove && gy == 0) word |= __ldg(&S.touchInTop[gx]);
        if (S.hasBelow && gy == S.latH - 1) word |= __ldg(&S.touchInBottom[gx]);
    }
    if (r2Point) {                                                  // tile (gx / 2, gy / 2): cell rows gy and gy + 1
        const int nbx = S.nbx;
        const uint16_t* cm = S.cellMask + (size_t)gy * nbx + (gx >> 4);
        m0 = __ldg(cm); m1 = __ldg(cm + nbx);
    }    // the total pointers of the CTA's final adds (thread p < YK_NPASS: pass p, thread YK_NPASS: R2)
    uint32_t* const finTot = threadIdx.x < YK_NPASS ? S.rgbTot[threadIdx.x] : nullptr;
    uint32_t* const finSup = threadIdx.x < YK_NPASS ? S.rgbSup[threadIdx.x] : nullptr;
    unsigned long long* const r2Tot = run.doR2 ? S.r2Tot : nullptr;
    unsigned long long* const r2Sup = run.doR2 ? S.r2Sup : nullptr;

    int key = -1, posK = 0;
    if (word != 0u && !(word & 0x80000000u))                        // touched, and not claimed by an earlier launch
        key = yk_owner_point(w, h, word, gx, gy, yk_pass_ids(run), posK);
    uint32_t *nib = nullptr, *tot = nullptr, *sup = nullptr;
    if (key >= 0) { nib = S.emitNib[key >> 24]; tot = S.rgbTot[key >> 24]; sup = S.rgbSup[key >> 24]; }
    int r2Key = -1;
    unsigned r2 = 0u;
    if (r2Point) {
        r2 = yk_r2_rule(m0, m1, gx >> 1);
        if (r2) r2Key = (int)((unsigned)((gy >> 1) * (w >> 3) + (gx >> 1)) / YK_EMIT_THREADS);
    }
    if (key >= 0) atomicOr(&nib[posK >> 5], 1u << (posK & 31));
    __syncthreads();
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
        else yk_rgb_add(tot, sup, key, rgbBytes);                   // another group of the same pass in this CTA
    }
    if (addR2) {
        if (sKey[YK_NPASS] == r2Key) atomicAdd(&sSum[YK_NPASS], r2Sum);
        else yk_r2_add(r2Tot, r2Sup, r2Key, r2Sum);
    }
    __syncthreads();
    if (threadIdx.x < YK_NPASS && sSum[threadIdx.x]) yk_rgb_add(finTot, finSup, sKey[threadIdx.x], sSum[threadIdx.x]);
    if (threadIdx.x == YK_NPASS && sSum[YK_NPASS]) yk_r2_add(r2Tot, r2Sup, sKey[YK_NPASS], sSum[YK_NPASS]);
}

// Block scan of the per-thread counts (c, d) plus the block sum of the per-thread base shares (pc, pd): returns the
// thread's exclusive offsets inside the block (offC, offD), and in every thread the block's base (baseC, baseD) and its own
// totals (totC, totD).
static __device__ __forceinline__ void yk_emit_scan(unsigned c, unsigned d, unsigned pc, unsigned pd, unsigned& offC, unsigned& offD,
                                                    unsigned& baseC, unsigned& baseD, unsigned& totC, unsigned& totD) {
    constexpr int NW = YK_EMIT_THREADS / 32;
    __shared__ unsigned sC[NW], sD[NW], sPC[NW], sPD[NW], sTot[4];
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
        if (lane < NW) { sC[lane] = ia - a; sD[lane] = ib - b; }
        if (lane == 31) { sTot[0] = ia; sTot[1] = ib; sTot[2] = bc; sTot[3] = bd; }
    }
    __syncthreads();
    offC = sC[warp] + ic - c; offD = sD[warp] + id - d;
    totC = sTot[0]; totD = sTot[1]; baseC = sTot[2]; baseD = sTot[3];
}

#ifndef YK_EMIT_LIST
#define YK_EMIT_LIST (4 * YK_EMIT_THREADS)      // corners a gradient group copies per round (a multiple of YK_EMIT_THREADS)
#endif
static_assert(YK_EMIT_LIST % YK_EMIT_THREADS == 0, "YK_EMIT_LIST: whole corners per thread");

// 512 threads (32 registers, 4 CTAs per SM): per pipelined step 41.2 us, 256 threads 41.3, 128 threads 42.3 (DESIGN.md §7,
// round-3 A/B log).  Both copies run over the whole CTA from a list in shared memory, and a thread issues the loads of a
// batch (2 corners, 4 chunks) before their stores: it waits for one round trip per batch, not one per byte or chunk (the
// stores may alias the loads as far as the compiler knows, so it would otherwise keep each load behind the previous store).
__global__ void __launch_bounds__(YK_EMIT_THREADS, 2048 / YK_EMIT_THREADS)
yk_k_emit(const YkSlotDev* __restrict__ slots, int slot0, YkRun run, int gradGroups, int r2Groups) {
    constexpr int T = YK_EMIT_THREADS;
    // gradient group: the lattice points of its corners (YK_EMIT_LIST per round); R2 group: tile << 2 | chunk of each of its
    // chunks (at most 4 T, 16 bits each)
    __shared__ uint32_t sList[YK_EMIT_LIST > 2 * T ? YK_EMIT_LIST : 2 * T];
    const YkSlotDev& S = slots[slot0 + blockIdx.y];
    const int tid = threadIdx.x;
    const int w = S.w, h = S.h;

    if ((int)blockIdx.x >= gradGroups) {
        // ---- DynamicTileCompressor streams: tiles in row-major order, 16 bytes per coded quadrant, 3 type bytes per coded tile
        const int grp = blockIdx.x - gradGroups, tilesW = w >> 3, nTiles = tilesW * (h >> 3);
        const int t0 = grp * T, t = t0 + tid;
        // this thread's share of the group's base: a group before it in its super-group, earlier super-groups
        unsigned long long pre = tid < grp % YK_SUPER ? S.r2Tot[grp - grp % YK_SUPER + tid] : 0ull;
        for (int s = tid; s < grp / YK_SUPER; s += T) pre += S.r2Sup[s];
        const unsigned c = t < nTiles ? yk_r2_count(S, t % tilesW, t / tilesW) : 0u;
        // the tile's type words, in flight during the scan (a tile that is not coded leaves them unused)
        uint32_t ty0 = 0u, ty1 = 0u, ty2 = 0u;
        if (t < nTiles) { ty0 = __ldg(&S.r2RawType[0][t]); ty1 = __ldg(&S.r2RawType[1][t]); ty2 = __ldg(&S.r2RawType[2][t]); }
        __shared__ const uint8_t* sRaw[3];                          // the plane pointers, loaded at entry (in registers they would spill)
        __shared__ uint8_t *sIdx[3], *sType[3];
        if (tid < 3) { sRaw[tid] = S.r2Raw[tid]; sIdx[tid] = S.r2Idx[tid]; sType[tid] = S.r2Type[tid]; }   // read after the scan's barriers
        const unsigned chunks = c >> 16;
        unsigned chunkOff, tileOff, chunkBase, tileBase, totC, totT;
        yk_emit_scan(chunks, chunks > 0, (unsigned)(pre >> 32), (unsigned)pre, chunkOff, tileOff, chunkBase, tileBase, totC, totT);
#ifdef YK_EMULATE
        if (tid == 0) assert(((unsigned long long)totC << 32 | totT) == S.r2Tot[grp]);     // yk_k_owner counted the same tiles
#endif
        if (grp == r2Groups - 1 && tid == 0) { S.hdr[YK_HD_R2_CHUNKS] = (int)(chunkBase + totC); S.hdr[YK_HD_R2_TILES] = (int)(tileBase + totT); }
        uint16_t* const sChunk = reinterpret_cast<uint16_t*>(sList);
        for (unsigned k = 0; k < chunks; k++) sChunk[chunkOff + k] = (uint16_t)(tid << 2 | k);
        if (chunks) {
            const size_t td = (size_t)(tileBase + tileOff) * 3;                                  // EC.cpp:8503-8505
            uint8_t *const d0 = sType[0] + td, *const d1 = sType[1] + td, *const d2 = sType[2] + td;
            d0[0] = (uint8_t)ty0; d0[1] = (uint8_t)(ty0 >> 8); d0[2] = (uint8_t)(ty0 >> 16);
            d1[0] = (uint8_t)ty1; d1[1] = (uint8_t)(ty1 >> 8); d1[2] = (uint8_t)(ty1 >> 16);
            d2[0] = (uint8_t)ty2; d2[1] = (uint8_t)(ty2 >> 8); d2[2] = (uint8_t)(ty2 >> 16);
        }
        __syncthreads();
        // the chunks of the three planes as one list of (plane, chunk) items, at most 4 per thread in a round
        const unsigned nItems = 3u * totC;
        for (unsigned i0 = tid; i0 < nItems; i0 += 4 * T) {
            uint4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const unsigned i = i0 + u * T;
                if (i < nItems) {
                    const unsigned p = i >= totC ? (i >= 2 * totC ? 2u : 1u) : 0u, e = sChunk[i - p * totC];
                    v[u] = __ldg(reinterpret_cast<const uint4*>(sRaw[p] + (size_t)(t0 + (e >> 2)) * 64) + (e & 3));
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const unsigned i = i0 + u * T;
                if (i < nItems) {
                    const unsigned p = i >= totC ? (i >= 2 * totC ? 2u : 1u) : 0u;
                    reinterpret_cast<uint4*>(sIdx[p])[chunkBase + i - p * totC] = v[u];
                }
            }
        }
        return;
    }

    // ---- rgbStream of one pass: CTA -> (pass position, group of 8 x YK_EMIT_THREADS tiles)
    const unsigned passIds = yk_pass_ids(run);
    int rp = 0, grp = blockIdx.x, nWords = 0, nSwzX = 0, nGroups = 0;
    YkGeomS g;
    for (;;) {
        g = yk_geom_s(yk_pass_at(passIds, rp));
        nSwzX = (w + (1 << g.lbw) - 1) >> g.lbw;
        nWords = (nSwzX * ((h + (1 << g.lbh) - 1) >> g.lbh) * g.bits) >> 3;
        nGroups = (nWords + T - 1) / T;
        if (grp < nGroups) break;
        grp -= nGroups; rp++;
    }
    const int pid = yk_pass_at(passIds, rp);
    unsigned pre = tid < grp % YK_SUPER ? S.rgbTot[pid][grp - grp % YK_SUPER + tid] : 0u;
    for (int s = tid; s < grp / YK_SUPER; s += T) pre += S.rgbSup[pid][s];
    const int wi = grp * T + tid;
    const uint32_t word = wi < nWords ? __ldg(&S.emitNib[pid][wi]) : 0u;
    const uint8_t* const lat = S.latRGB;
    const int latW = S.latW;
    // corner counts (the scan) and the byte base (the totals) come out separately: first = this thread's first corner in the group
    const unsigned mine = (unsigned)__popc(word);
    unsigned first, base, nCorners, unused0, unused1, unused2;
    yk_emit_scan(mine, 0u, pre, 0u, first, unused0, base, unused1, nCorners, unused2);
#ifdef YK_EMULATE
    if (tid == 0) assert(3u * nCorners == S.rgbTot[pid][grp]);                                  // yk_k_owner counted the same corners
#endif
    if (grp == nGroups - 1 && tid == 0) S.hdr[YK_HD_PASS0 + pid * YK_ST_STRIDE + YK_ST_RGBBYTES] = (int)(base + 3u * nCorners);
    uint8_t* const out = S.rgb[pid] + base;
    // the 8 tiles of a word share a swizzle block: invert the stream position once
    const int lbits = g.bits == 16 ? 4 : (g.bits == 32 ? 5 : 6);
    const int pos0 = wi * 8, blk = pos0 >> lbits, within0 = pos0 & (g.bits - 1);
    const int tprShift = g.lbw - g.shx;
    const int bys = blk / nSwzX, bxs = blk - bys * nSwzX;
    for (unsigned r0 = 0; r0 < nCorners; r0 += YK_EMIT_LIST) {
        // this thread's corners of the round, in stream order: ascending bit = tile, then TL, TR, BL, BR (EC.cpp:4115-4132)
        if (first < r0 + YK_EMIT_LIST && first + mine > r0) {
            uint32_t rest = word;
            for (unsigned i = first; rest && i < r0 + YK_EMIT_LIST; i++) {
                const int b = __ffs((int)rest) - 1;
                rest &= rest - 1u;
                if (i < r0) continue;
                const int within = within0 + (b >> 2), k = b & 3;
                const int gtx = (bxs << tprShift) + (within & ((1 << tprShift) - 1)), gty = (bys << (g.lbh - g.shy)) + (within >> tprShift);
                const int gx = ((gtx + (k & 1)) << g.shx) >> 2, gy = ((gty + (k >> 1)) << g.shy) >> 2;
                sList[i - r0] = (uint32_t)(gy * latW + gx);
            }
        }
        __syncthreads();
        const unsigned n = min(nCorners - r0, (unsigned)YK_EMIT_LIST);
        constexpr int K = YK_EMIT_LIST / T;
#pragma unroll
        for (int u0 = 0; u0 < K; u0 += 2) {                                                     // 2 corners in flight: 4 would spill
            uint8_t v[2][3];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const unsigned j = tid + (u0 + u) * T;
                if (u0 + u < K && j < n) { const uint8_t* sp = lat + (size_t)sList[j] * 3; v[u][0] = __ldg(sp); v[u][1] = __ldg(sp + 1); v[u][2] = __ldg(sp + 2); }
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const unsigned j = tid + (u0 + u) * T;
                if (u0 + u < K && j < n) { uint8_t* dp = out + (size_t)(r0 + j) * 3; dp[0] = v[u][0]; dp[1] = v[u][1]; dp[2] = v[u][2]; }
            }
        }
        if (r0 + YK_EMIT_LIST < nCorners) __syncthreads();                                      // the next round rewrites the list
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
