// yaik_b200 — auxiliary sm_100a kernels of the YAIK encoder-analysis stage (the hot path is yk_analyze.cu + yk_emit.cu):
//
//   yk_k_state        expands the compact masks into the reference's int32 state planes (compat download).
//   yk_k_r1_encode    DynamicTileEncode (EC.cpp:4365-4503, 747-1212), LUT search at 3/4 bits per pixel, on the colour planes
//                     or on the Y / reduced Co / Cg planes of the chroma front-end.
//   yk_k_chroma       RGB -> YCoCg + SampleDown of the chroma planes (Image.cpp:285-321, Plane.cpp:278-369).
//
// Reference line numbers are KLab/YAIK's encoder/EncoderContext.cpp ("EC.cpp") unless another file is named.
#include "yk_device.h"



struct YkGeomC { int shx, shy, bw, bh, bits; };
__constant__ YkGeomC yk_geom_tab[YK_NPASS] = YK_PASS_TABLE;
static __device__ __forceinline__ YkGeomC yk_geom(int pid) { return yk_geom_tab[pid]; }

// stream position (== bitmap bit index) of the tile at global tile coords (gtx, gty), EC.cpp:3801-3828, 4227-4234
static __device__ __forceinline__ int yk_tile_pos(const YkGeomC& g, int w, int gtx, int gty) {
    int x = gtx << g.shx, y = gty << g.shy;
    int nSwzX = (w + g.bw - 1) / g.bw;
    int gb = (y / g.bh) * nSwzX + (x / g.bw);
    return gb * g.bits + (((y % g.bh) >> g.shy) * (g.bw >> g.shx)) + ((x % g.bw) >> g.shx);
}

// ------------------------------------------------------------------------------------------------------------------
// pixel staging: 65x65 samples (the region plus the right/bottom corner row) of the three colour planes, clamped the
// way Plane::GetPixelValue clamps (framework.h:116-121), packed to bytes.
static __device__ __forceinline__ int yk_src(const YkSlotDev& S, int c, int x, int y) {
    x = min(x, S.w - 1);
    if (y >= S.h) {
        if (S.rowBelow[c])                                       // strip mode: the real row below (typed like the uploaded planes)
            return S.isU8 ? (int)__ldg(reinterpret_cast<const uint8_t*>(S.rowBelow[c]) + x) : __ldg(reinterpret_cast<const int32_t*>(S.rowBelow[c]) + x);
        y = S.h - 1;
    }
    return __ldg(S.plane[c] + (size_t)y * S.w + x);
}

static __device__ __forceinline__ unsigned yk_pack4(int4 v) {      // low bytes of four samples -> one word (3 PRMT)
    return __byte_perm(__byte_perm((unsigned)v.x, (unsigned)v.y, 0x0040), __byte_perm((unsigned)v.z, (unsigned)v.w, 0x0040), 0x5410);
}

static __device__ void yk_stage_pixels(const YkSlotDev& S, int X0, int Y0, uint8_t (*pix)[65 * YK_RS], unsigned& bad) {
    const int tid = threadIdx.x;
    const int w = S.w, h = S.h;
    for (int c = 0; c < 3; c++) {
        const int32_t* __restrict__ P = S.plane[c];
        int4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int ly = (tid >> 4) + 16 * k, lx = (tid & 15) * 4;
            int y = Y0 + ly, x = X0 + lx;
            if (y < h && x + 3 < w) {
                v[k] = __ldg(reinterpret_cast<const int4*>(P + (size_t)y * w + x));
            } else {
                v[k].x = yk_src(S, c, x, y); v[k].y = yk_src(S, c, x + 1, y);
                v[k].z = yk_src(S, c, x + 2, y); v[k].w = yk_src(S, c, x + 3, y);
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int ly = (tid >> 4) + 16 * k, lx = (tid & 15) * 4;
            bad |= (unsigned)(v[k].x | v[k].y | v[k].z | v[k].w);
            *reinterpret_cast<unsigned*>(&pix[c][ly * YK_RS + lx]) = yk_pack4(v[k]);
        }
        if (tid < 65) {                 // column 64
            int s = yk_src(S, c, X0 + 64, Y0 + tid);
            bad |= (unsigned)s;
            pix[c][tid * YK_RS + 64] = (uint8_t)s;
        } else if (tid < 65 + 64) {     // row 64
            int lx = tid - 65;
            int s = yk_src(S, c, X0 + lx, Y0 + 64);
            bad |= (unsigned)s;
            pix[c][64 * YK_RS + lx] = (uint8_t)s;
        }
    }
}

static __device__ __forceinline__ int yk_accept_bit(const YkSlotDev& S, int pid, const YkGeomC& g, int gtx, int gty) {
    if (gtx < 0 || gty < 0 || ((gtx + 1) << g.shx) > S.w || ((gty + 1) << g.shy) > S.h) return 0;
    int pos = yk_tile_pos(g, S.w, gtx, gty);
    return (S.bitmap[pid][pos >> 3] >> (pos & 7)) & 1;
}

// ------------------------------------------------------------------------------------------------------------------
// Compat download: expand the compact masks into the reference's int32 state planes (EncoderContext.h:300-323).
__global__ void __launch_bounds__(YK_THREADS)
yk_k_state(const YkSlotDev* __restrict__ slots, int slot, int32_t* smoothMap, int32_t* mipmapMask, int32_t* mappedRGB,
           int32_t* recon0, int32_t* recon1, int32_t* recon2) {
    __shared__ __align__(16) uint8_t pix[3][65 * YK_RS];
    __shared__ uint32_t sCell[16];
    const YkSlotDev& S = slots[slot];
    const int tid = threadIdx.x;
    const int w = S.w, h = S.h, nbx = S.nbx;
    const int bx = blockIdx.x % nbx, by = blockIdx.x / nbx;
    const int X0 = bx * YK_REGION, Y0 = by * YK_REGION;
    if (tid < 16) {
        int cy = (Y0 >> 2) + tid;
        sCell[tid] = (cy * 4 < h) ? S.cellMask[(size_t)cy * nbx + bx] : 0u;
    }
    unsigned bad = 0;
    if (recon0) yk_stage_pixels(S, X0, Y0, pix, bad);
    __syncthreads();
    const int tw16 = (w + 15) >> 4;
    for (int i = tid; i < 64 * 64; i += YK_THREADS) {
        const int lx = i & 63, ly = i >> 6, x = X0 + lx, y = Y0 + ly;
        if (x >= w || y >= h) continue;
        const bool claimed = (sCell[ly >> 2] >> (lx >> 2)) & 1u;
        const size_t o = (size_t)y * w + x;
        if (smoothMap) smoothMap[o] = claimed ? 255 : 0;
        if (mipmapMask) {
            int mv = 255;
            if (S.alphaValid && !S.alphaReset && !S.alphaKept[(size_t)(y >> 4) * tw16 + (x >> 4)]) mv = 0;    // EC.cpp:394-414
            if (claimed) mv = 0;                                                                               // EC.cpp:4035
            mipmapMask[o] = mv;
        }
        if (recon0) { recon0[o] = 0; recon1[o] = 0; recon2[o] = 0; }
    }
    if (mappedRGB) {
        const int xMax = (bx == nbx - 1) ? 65 : 64, yMax = (by == S.nby - 1) ? 65 : 64;
        for (int i = tid; i < 65 * 65; i += YK_THREADS) {
            const int lx = i % 65, ly = i / 65, x = X0 + lx, y = Y0 + ly;
            if (lx >= xMax || ly >= yMax || x > w || y > h) continue;
            int v = 0;
            if (!(x & 3) && !(y & 3)) v = S.touchMap[(size_t)(y >> 2) * S.latW + (x >> 2)] ? 255 : 0;
            mappedRGB[(size_t)y * (w + 1) + x] = v;
        }
    }
    if (!recon0) return;
    __syncthreads();
    // recon = Round6P family, rounded variant, of every accepted tile; later passes overwrite earlier ones
    // (EC.cpp:3969-3971, 4096-4104), passes in Convert()'s order
    int32_t* rec[3] = { recon0, recon1, recon2 };
    for (int pid = 0; pid < YK_NPASS; pid++) {
        const YkGeomC g = yk_geom(pid);
        const int tw = 1 << g.shx, th = 1 << g.shy, N = tw * th, NX = 64 / tw;
        for (int i = tid; i < 64 * 64; i += YK_THREADS) {
            const int lx = i & 63, ly = i >> 6;
            const int tx = lx / tw, ty = ly / th;
            if (!yk_accept_bit(S, pid, g, bx * NX + tx, by * (64 / th) + ty)) continue;
            const int lx0 = tx * tw, ly0 = ty * th, dx = lx - lx0, dy = ly - ly0;
            for (int c = 0; c < 3; c++) {
                const uint8_t* p = pix[c];
                int tl = yk_round6p(p[ly0 * YK_RS + lx0]), tr = yk_round6p(p[ly0 * YK_RS + lx0 + tw]);
                int bl = yk_round6p(p[(ly0 + th) * YK_RS + lx0]), br = yk_round6p(p[(ly0 + th) * YK_RS + lx0 + tw]);
                int s = (tl * (tw - dx) + tr * dx) * (th - dy) + (bl * (tw - dx) + br * dx) * dy;
                rec[c][(size_t)(Y0 + ly) * w + X0 + lx] = (s + N / 2 - 1) / N;
            }
        }
        __syncthreads();
    }
}


// ------------------------------------------------------------------------------------------------------------------
// Range stage R1: DynamicTileEncode (EC.cpp:4365-4503) = LeftRightOrder walk (framework.h:228-256, yk_r1_walk) over the
// 8-aligned bound box, GetMinMax_Y (Plane.cpp:489-587) and GetTileDynamic_Y (EC.cpp:747-1212) per 8x8 block.
// valid pixel = mipmapMask != 0 && smoothMap == 0 (Plane.cpp:525-527).

// block-wide exclusive scan of one int per thread (used by the R1 offset scan)
static __device__ int yk_block_exclusive(int v, int* sWarp, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(YK_FULL, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) sWarp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int x = lane < nw ? sWarp[lane] : 0, xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(YK_FULL, xi, d); if (lane >= d) xi += t; }
        sWarp[lane] = xi - x;
        if (lane == 31) sWarp[32] = xi;
    }
    __syncthreads();
    total = sWarp[32];
    const int r = sWarp[warp] + inc - v;
    __syncthreads();
    return r;
}

// Two launches code one plane (a colour plane, or Y / reduced Co / Cg of the chroma front-end) or the three
// full-resolution colour planes R, G, B, which share their geometry and validity:
//   yk_k_r1_offsets   one thread per block of the walk: which pixel pairs of the block are coded (that only depends on
//                     the alpha / claimed-cell masks, not on the samples), a block scan + one decoupled look-back per
//                     YK_R1_UNIT blocks give the nibble / tile-def offsets - the same for every plane - and the blocks
//                     that hold valid pixels are listed in walk order {x | y << 16, pairs, nibble offset}.
//   yk_k_r1_encode    one plane: warps take listed blocks with a grid stride and code them independently of each other
//                     (no block barrier, no waiting): min / max, table, mode search, ordered error sums, output at the
//                     final stream position.
//   yk_k_r1_encode3   the three colour planes: a warp codes the three planes of a listed block in one go.
// Both encode kernels code a (block, plane) with the same steps (yk_r1_load2 .. yk_r1_output below).
//
// lut: [64 base6][YK_R1_R7MAX range7][YK_R1_LUT_INTS] ints.  [0,72) = the six LUTs (16,16,16,8,8,8 entries) of DynamicTile::buildTable
// (EC.cpp:625-699); [72,144) = their decision thresholds, same layout.  Every LUT is non-decreasing, so the reference's
// "first strict minimum of |entry - value|" scan (EC.cpp:873-881) picks entry n over all earlier ones exactly when
// value > floor((L[n-1] + L[n]) / 2) with L[n] > L[n-1]; a repeated entry is never picked and inherits the threshold of
// the next distinct one (INT_MAX if none), which keeps the thresholds non-decreasing: code = #{n >= 1 : value > thr[n]}
// = the largest n with value > thr[n] (binary search).
// rtab: [64][128 range7 < 128][6 modes][384] u16 = code << 8 | LUT entry that search picks, for every value 0..383 (the
// domain of the reference's tables: samples -128..255, shifted by 128 when the block's minimum is negative), built on
// the host from the same thresholds: the per-pixel, per-mode work of the mode search is one 16-bit load.
#define YK_R1_THREADS 128           // CTA size of the encode kernels

// Validity of one full-resolution pixel as DynamicTileEncode sees it: mipmapMask != 0 (kept by the alpha stage) and
// smoothMap == 0 (its 4x4 cell not claimed by a gradient tile).
static __device__ __forceinline__ bool yk_r1_mask_at(const YkSlotDev& S, bool maskActive, int fx, int fy) {
    return !(maskActive && !S.alphaKept[(size_t)(fy >> 4) * ((S.w + 15) >> 4) + (fx >> 4)]);
}
static __device__ __forceinline__ bool yk_r1_smooth_at(const YkSlotDev& S, int fx, int fy) {
    const int cx = fx >> 2;
    return (S.cellMask[(size_t)(fy >> 2) * S.nbx + (cx >> 4)] >> (cx & 15)) & 1u;
}
// mipmapMask != 0 at linear index i of the full-size mask plane
static __device__ __forceinline__ bool yk_r1_valid_at(const YkSlotDev& S, bool maskActive, size_t i) {
    const int fx = (int)(i % (size_t)S.w), fy = (int)(i / (size_t)S.w);
    return yk_r1_mask_at(S, maskActive, fx, fy) && !yk_r1_smooth_at(S, fx, fy);
}
// unclaimed-and-kept 4x4 cells of the 8x8 block at (x, y): bit0 TL, bit1 TR, bit2 BL, bit3 BR
static __device__ __forceinline__ unsigned yk_r1_cells(const YkSlotDev& S, bool maskActive, int x, int y) {
    if (!yk_r1_mask_at(S, maskActive, x, y)) return 0u;
    const int cx = x >> 2, cy = y >> 2;
    const unsigned r0 = S.cellMask[(size_t)cy * S.nbx + (cx >> 4)], r1 = S.cellMask[(size_t)(cy + 1) * S.nbx + (cx >> 4)];
    return (~(((r0 >> (cx & 15)) & 3u) | (((r1 >> (cx & 15)) & 3u) << 2))) & 15u;
}

// Block b0 + i of the walk is (cx + 8*(j % nbw), cy + 8*(j / nbw)), j = b0 + i, in image coordinates.  Block sizes: the reference compares with the
// constraint's width / height, not its right / bottom edge, and falls back to x % 8 (framework.h:251-252) - 0 for the
// full-resolution planes (x + 8 > cw empties the block), possibly 4 for a reduced chroma plane whose box starts on an
// odd multiple of 4.
struct YkR1Block { int x, y, rw, rh; };
static __device__ __forceinline__ YkR1Block yk_r1_block(const YkR1Walk& G, int i) {
    YkR1Block b;
    const int j = G.b0 + i;
    b.x = G.cx + 8 * (j % G.nbw); b.y = G.cy + 8 * (j / G.nbw);
    b.rw = (b.x + 8 > G.cw) ? (b.x & 7) : 8;
    b.rh = (b.y + 8 > G.ch) ? (b.y & 7) : 8;
    return b;
}

// float(d) / float(o), correctly rounded, for the small integers of this stage: with r = RN(1 / o) the residual
// correction below reproduces IEEE division for all 1 <= d, o <= 2048 (checked exhaustively on the host, DESIGN.md);
// anything larger takes the division itself.
static __device__ __forceinline__ float yk_r1_quot(int d, float fo, float r) {
    const float fd = __int2float_rn(d);
    const float q0 = __fmul_rn(fd, r);
    return __fmaf_rn(__fmaf_rn(-q0, fo, fd), r, q0);                // r == 0 (a dropped term) gives exactly +0
}

struct YkR1Item { unsigned xy, pairs, nibOff, pad; };        // one listed block: see yk_k_r1_offsets

// the launch's walk and whether mipmapMask holds the alpha stage's rejection
struct YkR1Geom { YkR1Walk walk; int maskActive; };
static __device__ YkR1Geom yk_r1_geometry(const YkSlotDev& S, const YkR1Launch& LP) {
    YkR1Geom G;
    G.walk = LP.walk;
    G.maskActive = S.alphaValid && !S.alphaReset;
    if (LP.fromHdr) {
        // the bound box of the alpha stage straight from the image header the analysis kernel has just written
        // (CheckMipmapMask's full image without an alpha stage)
        int box[4] = { 0, 0, S.w, S.h };
        G.maskActive = 0;
        if (LP.useAlpha && S.nPlanes == 4 && yk_alpha_box(S.hdr, S.w, box)) G.maskActive = !yk_box_is_image(box, S.w, S.imgH);
        G.walk = yk_r1_walk(box, LP.ph, LP.shX, LP.shY);
    }
    return G;
}

__global__ void __launch_bounds__(YK_R1_UNIT)
yk_k_r1_offsets(const YkSlotDev* __restrict__ slots, int slot, const YkR1Launch LP) {
    __shared__ int sWarp[33];
    __shared__ int sUnit;
    __shared__ unsigned sBase[2];
    __shared__ YkR1Geom sG;
    const YkSlotDev& S = slots[slot];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool reduced = (LP.shX | LP.shY) != 0;
    unsigned long long* status = S.r1Status;
    if (tid == 0) {
        const YkR1Geom G = yk_r1_geometry(S, LP);
        sG = G;
        const int nU = (G.walk.nBlocks + YK_R1_UNIT - 1) / YK_R1_UNIT;
        sUnit = (int)atomicAdd(reinterpret_cast<unsigned*>(&status[nU]), 1u);
    }
    __syncthreads();
    const YkR1Walk G = sG.walk;
    const bool maskActive = sG.maskActive != 0;
    const int nUnits = (G.nBlocks + YK_R1_UNIT - 1) / YK_R1_UNIT;
    const int u = sUnit;
    if (u >= nUnits) {                                            // launched for the largest possible box
        if (nUnits == 0 && u == 0 && tid == 0) {
            for (int j = 0; j < LP.nJobs; j++) { S.hdr[YK_HD_R1_NIB0 + LP.job[j].out] = 0; S.hdr[YK_HD_R1_DEF0 + LP.job[j].out] = 0; }
        }
        return;
    }
    // ---- count: which pixel pairs of my block are coded (EC.cpp:826-861; the 2x2 / 2x1 / 1x2 mask samples a reduced
    // pixel covers lie in one 16x16 alpha tile, so "all of them" is the top-left one)
    const int i = u * YK_R1_UNIT + tid;
    unsigned pairs = 0;
    YkR1Block b = { 0, 0, 0, 0 };
    if (i < G.nBlocks) {
        b = yk_r1_block(G, i);
        if (!reduced) {
            // the geometry is the image's; the masks, and the samples the encode kernels read from the list entry, are
            // the strip's rows (y0 == 0 for a whole image)
            b.y -= S.y0;
            if (b.rw == 8 && b.rh == 8 && b.x + 8 <= S.w && b.y + 8 <= S.h) {
                const unsigned cells = yk_r1_cells(S, maskActive, b.x, b.y);
                pairs = ((cells & 1u) ? 0x00003333u : 0u) | ((cells & 2u) ? 0x0000CCCCu : 0u) | ((cells & 4u) ? 0x33330000u : 0u) | ((cells & 8u) ? 0xCCCC0000u : 0u);
            }
        } else {
            for (int r = 0; r < b.rh; r++)
                for (int p = 0; 2 * p < b.rw; p++) {
                    const int fx = (b.x + 2 * p) << LP.shX, fy = (b.y + r) << LP.shY;
                    if (yk_r1_mask_at(S, maskActive, fx, fy) && !yk_r1_smooth_at(S, fx, fy)) pairs |= 1u << (4 * r + p);
                }
        }
    }
    const int n = 2 * __popc(pairs);
    // ---- offsets: pixels in the low 16 bits (<= 64 * YK_R1_UNIT per unit), blocks with pixels above
    int tot;
    const int ex = yk_block_exclusive(n | ((n > 0) << 16), sWarp, tot);
    if (warp == 0) {
        const unsigned long long base = yk_lookback64(status, u, (unsigned)(tot & 0xFFFF), (unsigned)(tot >> 16));
        if (lane == 0) {
            sBase[0] = (unsigned)(base >> 32); sBase[1] = (unsigned)base;
            if (u == nUnits - 1)
                for (int j = 0; j < LP.nJobs; j++) {
                    S.hdr[YK_HD_R1_NIB0 + LP.job[j].out] = (int)(base >> 32) + (tot & 0xFFFF);
                    S.hdr[YK_HD_R1_DEF0 + LP.job[j].out] = (int)(unsigned)base + (tot >> 16);
                }
        }
    }
    __syncthreads();
    if (n > 0) {
        YkR1Item it;
        it.xy = (unsigned)b.x | ((unsigned)b.y << 16); it.pairs = pairs; it.nibOff = sBase[0] + (unsigned)(ex & 0xFFFF); it.pad = (unsigned)b.rw | ((unsigned)b.rh << 8);
        reinterpret_cast<uint4*>(S.r1List)[sBase[1] + (unsigned)(ex >> 16)] = make_uint4(it.xy, it.pairs, it.nibOff, it.pad);
    }
}

// ---- The steps of coding one (listed block, plane), shared by both encode kernels.  Lane l holds the pixel pair
// (c0, c0 + 1) = (2 (l & 3), 2 (l & 3) + 1) of row r = l >> 2 of the block.  A plane's state between the steps is one
// word: b6 | r7 << 8 | sgn << 16 | tabled << 24.

// the lane's two samples at (x, y) of a plane of width pw, u8 or int32
static __device__ __forceinline__ void yk_r1_load2(const YkR1Args& A, int pw, int x, int y, int& v0, int& v1) {
    if (A.srcU8) {
        const unsigned short two = __ldg(reinterpret_cast<const unsigned short*>(A.srcU8 + (size_t)y * A.pitchU8 + x));
        v0 = two & 255; v1 = two >> 8;
    } else {
        const int2 p = __ldg(reinterpret_cast<const int2*>(A.src + (size_t)y * pw + x));
        v0 = p.x; v1 = p.y;
    }
}
// list entry `at` and, when `samples` is set and the lane's pair is coded, the pair's samples of the first NP planes:
// fetched while the warp codes the entry before
template <int NP>
static __device__ __forceinline__ void yk_r1_fetch(const YkSlotDev& S, const YkR1Launch& LP, int at, int nList, bool samples, uint4& item, int (&v)[NP][2]) {
    if (at >= nList) return;
    const int lane = threadIdx.x & 31;
    item = __ldg(reinterpret_cast<const uint4*>(S.r1List) + at);
    const bool on = samples && ((item.y >> lane) & 1u);
    const int x = (item.x & 0xFFFF) + (lane & 3) * 2, y = (item.x >> 16) + (lane >> 2);
#pragma unroll
    for (int j = 0; j < NP; j++) {
        v[j][0] = 0; v[j][1] = 0;
        if (on) yk_r1_load2(LP.job[j], LP.pw, x, y, v[j][0], v[j][1]);
    }
}

// min / max of the block over the samples whose flag is set (Plane::GetMinMax_Y, Plane.cpp:489-587), the sign shift
// (EC.cpp:764-768) and the table index (DynamicTile::buildTable, EC.cpp:635-650); o0 / o1 become the shifted samples
struct YkR1Tab { int b6, r7, sgn; bool tabled; };
static __device__ __forceinline__ YkR1Tab yk_r1_table(int& o0, int& o1, bool m0, bool m1, const short* __restrict__ r7tab) {
    int mn = __reduce_min_sync(YK_FULL, min(m0 ? o0 : INT_MAX, m1 ? o1 : INT_MAX));
    int mx = __reduce_max_sync(YK_FULL, max(m0 ? o0 : INT_MIN, m1 ? o1 : INT_MIN));
    if (mn == INT_MAX) { mn = 0; mx = 0; }                                 // Plane.cpp:579-585
    int sgn = 0;
    if (mn < 0) { mn += 128; mx += 128; sgn = 128; }
    mn = min(max(mn, 0), 255); mx = min(max(mx, mn), 255);
    const int m = min(mn, YK_R1_BASE_MAX);
    const int diff = max(mx - m, 16);
    const int b6 = (m * 63 + YK_R1_BASE_MAX / 2) / YK_R1_BASE_MAX;
    // ((max(diff,32) - 32) * 127 + scale - 1) / scale, scale = 223 - BN (EC.cpp:643-650): 0..170 for every reachable (b6, diff)
    const int r7 = __ldg(r7tab + b6 * YK_R1_R7_ROW + (max(diff, 32) - 32));
    o0 += sgn; o1 += sgn;
    // the per-value table covers range codes below 128, bases below 63 (the other LUTs have entries above 255: reference
    // quirks) and samples 0..383; anything else takes the search and the division themselves
    const bool tabled = r7 < YK_R1_RTAB_R7 && b6 < 63 && __all_sync(YK_FULL, (unsigned)o0 < (unsigned)YK_R1_RTAB_VALUES && (unsigned)o1 < (unsigned)YK_R1_RTAB_VALUES);
    return YkR1Tab{ b6, r7, sgn, tabled };
}
// the state word that carries a plane from the mode search to its output: b6 | r7 << 8 | sgn << 16 | tabled << 24
static __device__ __forceinline__ int yk_r1_pack(const YkR1Tab& t) { return t.b6 | (t.r7 << 8) | (t.sgn << 16) | ((int)t.tabled << 24); }

static __device__ __forceinline__ int yk_r1_off(int mode) { return mode < 3 ? 16 * mode : 48 + 8 * (mode - 3); }    // LUT `mode` in an lut row
static __device__ __forceinline__ const int* yk_r1_lut(const int* __restrict__ lut, int b6, int r7) {
    return lut + (size_t)(b6 * YK_R1_R7MAX + min(r7, YK_R1_R7MAX - 1)) * YK_R1_LUT_INTS;
}
static __device__ __forceinline__ const unsigned short* yk_r1_rtab(const unsigned short* __restrict__ rtab, int b6, int r7) {     // tabled planes
    return rtab + (size_t)(b6 * YK_R1_RTAB_R7 + r7) * (6 * YK_R1_RTAB_VALUES);
}
// the codes of o0 / o1 in LUT `mode` of the lut row T: the largest n with value > threshold[n]
static __device__ __forceinline__ void yk_r1_search(const int* T, int mode, int o0, int o1, int& g0, int& g1) {
    const int off = yk_r1_off(mode);
    g0 = 0; g1 = 0;
    for (int st = (mode < 3 ? 8 : 4); st > 0; st >>= 1) {
        if (o0 > __ldg(T + 72 + off + g0 + st)) g0 += st;
        if (o1 > __ldg(T + 72 + off + g1 + st)) g1 += st;
    }
}

// relative error terms of the lane's pair, float32 (EC.cpp:884-886): float(|entry - value|) / float(value) for the modes
// from startMode on, into term[mode][pixel].  Invalid pixels and zero samples add +0.0f, which leaves the sum unchanged:
// their reciprocal is set to zero here, and a zero difference gives a zero quotient by itself.
static __device__ __forceinline__ void yk_r1_terms(float (*term)[64], const YkR1Tab& t, int o0, int o1, bool valid, int startMode,
                                                   const int* __restrict__ lut, const unsigned short* __restrict__ rtab) {
    const int lane = threadIdx.x & 31;
    const bool use0 = valid && o0 != 0, use1 = valid && o1 != 0;
    const float f0 = __int2float_rn(use0 ? o0 : 1), f1 = __int2float_rn(use1 ? o1 : 1);
    const float rc0 = use0 ? __frcp_rn(f0) : 0.0f, rc1 = use1 ? __frcp_rn(f1) : 0.0f;
    if (t.tabled) {
        const unsigned short* RT = yk_r1_rtab(rtab, t.b6, t.r7);
#pragma unroll
        for (int mode = 0; mode < 6; mode++) {
            if (mode < startMode) continue;
            const int L0 = __ldg(RT + mode * YK_R1_RTAB_VALUES + o0) & 255, L1 = __ldg(RT + mode * YK_R1_RTAB_VALUES + o1) & 255;
            *reinterpret_cast<float2*>(&term[mode][2 * lane]) = make_float2(yk_r1_quot(abs(L0 - o0), f0, rc0), yk_r1_quot(abs(L1 - o1), f1, rc1));
        }
    } else {
        const int* T = yk_r1_lut(lut, t.b6, t.r7);
#pragma unroll 1
        for (int mode = startMode; mode < 6; mode++) {
            int g0, g1;
            yk_r1_search(T, mode, o0, o1, g0, g1);
            const int off = yk_r1_off(mode);
            const int d0 = abs(__ldg(T + off + g0) - o0), d1 = abs(__ldg(T + off + g1) - o1);
            term[mode][2 * lane] = (use0 && d0 != 0) ? __fdiv_rn(__int2float_rn(d0), f0) : 0.0f;
            term[mode][2 * lane + 1] = (use1 && d1 != 0) ? __fdiv_rn(__int2float_rn(d1), f1) : 0.0f;
        }
    }
}

// the error of one (plane, mode): its 64 terms summed in row-major pixel order, as the reference sums (float addition is
// not associative, so one lane per sum).  float4 group q = pixels 4q .. 4q + 3 = row q >> 1, left (q even) or right half:
// a quadrant without coded pairs holds +0.0f only and is skipped, which is exact since the sum never is -0.0f.
static __device__ __forceinline__ float yk_r1_sum(const float* terms, unsigned pairs) {
    const float4* P = reinterpret_cast<const float4*>(terms);
    float err = 0.0f;
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const unsigned hm = (pairs >> (16 * half)) & 0xFFFFu;
        if (hm) {
            const bool Lq = (hm & 0x3333u) != 0u, Rq = (hm & 0xCCCCu) != 0u;
            if (Lq && Rq) {
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    const float4 t = P[8 * half + q];
                    err = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(err, t.x), t.y), t.z), t.w);
                }
            } else {
                const float4* Q = P + 8 * half + (Rq ? 1 : 0);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const float4 t = Q[2 * q];
                    err = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(err, t.x), t.y), t.z), t.w);
                }
            }
        }
    }
    return err;
}

// the best mode among the errors of the lanes that are `mine`: the highest such lane that holds their minimum, as `<=`
// lets later modes win ties (EC.cpp:897-905).  Sums can be negative on signed chroma planes: compare through the
// order-preserving map of the bit patterns (-0 counted as +0, as `<=` does).
static __device__ __forceinline__ int yk_r1_best(float err, bool mine) {
    const unsigned eraw = __float_as_uint(__fadd_rn(err, 0.0f));
    const unsigned ebits = mine ? (eraw ^ ((eraw >> 31) ? 0xFFFFFFFFu : 0x80000000u)) : 0xFFFFFFFFu;
    const unsigned emin = __reduce_min_sync(YK_FULL, ebits);
    return 31 - __clz((int)__ballot_sync(YK_FULL, mine && ebits == emin));
}

// output in the chosen mode: the codes of a valid lane's pair (from the per-value table again, or the search), their
// nibble byte at nibble n0 (even: the two nibbles share a byte), the optional write-back of the pair at (x, y) of a
// plane reduced by shX / shY, and the tile def of list entry k
static __device__ __forceinline__ void yk_r1_output(const YkSlotDev& S, const YkR1Args& A, int shX, int shY, int meta, int mode, bool valid,
                                                    int o0, int o1, int n0, int x, int y, int k,
                                                    const int* __restrict__ lut, const unsigned short* __restrict__ rtab) {
    const int b6 = meta & 255, r7 = (meta >> 8) & 255;
    if (valid) {
        const int* T = yk_r1_lut(lut, b6, r7);
        int c0v, c1v;
        if ((meta >> 24) & 1) {
            const unsigned short* RT = yk_r1_rtab(rtab, b6, r7) + mode * YK_R1_RTAB_VALUES;
            c0v = __ldg(RT + o0) >> 8; c1v = __ldg(RT + o1) >> 8;
        } else {
            yk_r1_search(T, mode, o0, o1, c0v, c1v);
        }
        reinterpret_cast<uint8_t*>(S.r1Nib[A.out])[n0 >> 1] = (uint8_t)(c0v | (c1v << 4));   // low nibble first, EC.cpp:1180-1184
        if (A.dst) {
            // EC.cpp:4441-4502: chroma blocks with a negative minimum go back minus 128; reduced planes are written at
            // their top-left full-size position only ("interpolation comes later")
            const int off = yk_r1_off(mode), offset = (A.chroma && ((meta >> 16) & 255)) ? -128 : 0;
            int* d = A.dst + (size_t)(y << shY) * S.w + (x << shX);
            d[0] = __ldg(T + off + c0v) + offset; d[1 << shX] = __ldg(T + off + c1v) + offset;
        }
    }
    if ((threadIdx.x & 31) == 0) S.r1Defs[A.out][k] = (uint16_t)((mode << 13) | (r7 << 7) | b6);    // EncodeTileType, YAIK_private.h:358
}

// One plane (nJobs == 1): a warp takes a listed block and codes it.
#define YK_R1_MINB 9                // resident CTAs per SM the register budget is set for
#define YK_R1_CAP 12                // CTAs per SM at most in a launch
__global__ void __launch_bounds__(YK_R1_THREADS, YK_R1_MINB)
yk_k_r1_encode(const YkSlotDev* __restrict__ slots, int slot, const YkR1Launch LP, const int* __restrict__ lut, const unsigned short* __restrict__ rtab, const short* __restrict__ r7tab) {
    __shared__ __align__(16) float sTerm[YK_R1_THREADS / 32][6][64];
    const YkSlotDev& S = slots[slot];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const YkR1Args& A = LP.job[0];
    const bool reduced = (LP.shX | LP.shY) != 0;
    const bool maskActive = reduced ? (yk_r1_geometry(S, LP).maskActive != 0) : false;      // only the reduced planes look at the masks again
    const int nList = __ldg(&S.hdr[YK_HD_R1_DEF0 + A.out]);                                 // written by yk_k_r1_offsets
    const int r = lane >> 2, c0 = (lane & 3) * 2;
    const int startMode = LP.mode3 ? 3 : 0;
    const bool summing = lane >= startMode && lane < 6;                                    // the lane that sums mode `lane`
    float (*term)[64] = sTerm[warp];
    // the next block's list entry and (full-resolution planes) its samples are fetched while the current one is coded
    const int stride = gridDim.x * (YK_R1_THREADS / 32);
    int k = blockIdx.x * (YK_R1_THREADS / 32) + warp;
    uint4 nItem = make_uint4(0u, 0u, 0u, 0u);
    int nv[1][2] = { { 0, 0 } };
    yk_r1_fetch(S, LP, k, nList, !reduced, nItem, nv);
    for (; k < nList; k += stride) {
        const uint4 item = nItem;
        int o0 = nv[0][0], o1 = nv[0][1];
        yk_r1_fetch(S, LP, k + stride, nList, !reduced, nItem, nv);
        const int x = item.x & 0xFFFF, y = item.x >> 16;
        const bool valid = (item.y >> lane) & 1u;
        // ---- min / max of the block.  Full resolution: over the coded pixels.  Reduced planes: over "not smooth and any
        // covered mask sample set", where the reference addresses the full-size mask with the REDUCED plane's width as
        // row stride (Plane.cpp:516, 538-553) - restated literally.
        bool m0 = valid, m1 = valid;
        if (reduced) {
            const int brw = item.w & 255, brh = (item.w >> 8) & 255;
            m0 = m1 = false;
            if (r < brh && c0 < brw) {
#pragma unroll
                for (int q = 0; q < 2; q++) {
                    const size_t vi = ((size_t)(x + c0 + q) << LP.shX) + (size_t)((y + r) << LP.shY) * LP.pw;
                    const int W = S.w;
                    // every covered sample is a mipmapMask value: kept by the alpha stage AND not claimed by a gradient
                    // tile (FittingQuadSmooth zeroes the mask over accepted tiles, EC.cpp:4035); with the reduced width as
                    // row stride the samples of the second row lie in another cell than vi
                    bool any = yk_r1_valid_at(S, maskActive, vi);
                    if (LP.shX) any |= yk_r1_valid_at(S, maskActive, vi + 1);
                    if (LP.shY) any |= yk_r1_valid_at(S, maskActive, vi + LP.pw);
                    if (LP.shX && LP.shY) any |= yk_r1_valid_at(S, maskActive, vi + LP.pw + 1);
                    const bool ok = any && !yk_r1_smooth_at(S, (int)(vi % W), (int)(vi / W));
                    if (q) m1 = ok; else m0 = ok;
                }
            }
            if (valid || m0 || m1) yk_r1_load2(A, LP.pw, x + c0, y + r, o0, o1);
        }
        const YkR1Tab t = yk_r1_table(o0, o1, m0, m1, r7tab);
        yk_r1_terms(term, t, o0, o1, valid, startMode, lut, rtab);
        __syncwarp();
        const int best = yk_r1_best(summing ? yk_r1_sum(term[lane], item.y) : 0.0f, summing);
        __syncwarp();                                                           // the terms are rewritten by the next block
        const int n0 = (int)item.z + 2 * __popc(item.y & ((1u << lane) - 1u));   // coded pairs == lanes with pixels
        yk_r1_output(S, A, LP.shX, LP.shY, yk_r1_pack(t), best, valid, o0, o1, n0, x + c0, y + r, k, lut, rtab);
    }
}

// The three full-resolution colour planes of one launch (nJobs == 3, the fused yk_analyze path): a warp takes a listed
// block and codes its three planes in one go.  What a block costs besides its per-pixel work is shared by the planes
// (list entry, geometry, validity ballots), and the ordered error sums - 64 dependent float adds that one lane per mode
// has to do whatever the other lanes are up to - run for the 18 (plane, mode) pairs side by side in 18 lanes.
#define YK_R1_MINB3 8
#define YK_R1_CAP3 8
__global__ void __launch_bounds__(YK_R1_THREADS, YK_R1_MINB3)
yk_k_r1_encode3(const YkSlotDev* __restrict__ slots, int slot, const YkR1Launch LP, const int* __restrict__ lut, const unsigned short* __restrict__ rtab, const short* __restrict__ r7tab) {
    __shared__ __align__(16) float sTerm[YK_R1_THREADS / 32][3][6][64];
    const YkSlotDev& S = slots[slot];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nList = __ldg(&S.hdr[YK_HD_R1_DEF0 + LP.job[0].out]);                         // written by yk_k_r1_offsets
    const int r = lane >> 2, c0 = (lane & 3) * 2;
    const int startMode = LP.mode3 ? 3 : 0;
    float (*term)[6][64] = sTerm[warp];
    // the lane that sums (plane sj, mode sm)
    const int sj = lane / 6, sm = lane - 6 * sj;
    const bool summing = lane < 18 && sm >= startMode;
    const int stride = gridDim.x * (YK_R1_THREADS / 32);
    int k = blockIdx.x * (YK_R1_THREADS / 32) + warp;
    uint4 nItem = make_uint4(0u, 0u, 0u, 0u);
    int nv[3][2] = { { 0, 0 }, { 0, 0 }, { 0, 0 } };
    yk_r1_fetch(S, LP, k, nList, true, nItem, nv);
    for (; k < nList; k += stride) {
        const uint4 item = nItem;
        int o[3][2];
#pragma unroll
        for (int j = 0; j < 3; j++) { o[j][0] = nv[j][0]; o[j][1] = nv[j][1]; }
        yk_r1_fetch(S, LP, k + stride, nList, true, nItem, nv);
        const int x = item.x & 0xFFFF, y = item.x >> 16;
        const bool valid = (item.y >> lane) & 1u;
        int meta[3];
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const YkR1Tab t = yk_r1_table(o[j][0], o[j][1], valid, valid, r7tab);
            meta[j] = yk_r1_pack(t);
            yk_r1_terms(term[j], t, o[j][0], o[j][1], valid, startMode, lut, rtab);
        }
        __syncwarp();
        const float err = summing ? yk_r1_sum(term[sj][sm], item.y) : 0.0f;
        int best[3];
#pragma unroll
        for (int j = 0; j < 3; j++) best[j] = yk_r1_best(err, summing && sj == j) - 6 * j;
        __syncwarp();                                                           // the terms are rewritten by the next block
        const int n0 = (int)item.z + 2 * __popc(item.y & ((1u << lane) - 1u));   // coded pairs == lanes with pixels
#pragma unroll
        for (int j = 0; j < 3; j++) yk_r1_output(S, LP.job[j], 0, 0, meta[j], best[j], valid, o[j][0], o[j][1], n0, x + c0, y + r, k, lut, rtab);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Chroma front-end (SURVEY.md 8f row 3): Image::ConvertToRGB2YCoCg (Image.cpp:285-321, RGBtoYCoCg EC.cpp:53-67) fused
// with EncoderContext::chromaReduction (EC.cpp:2770-2782) = Plane::SampleDown (Plane.cpp:278-369) of Co and of Cg.
// One thread per 2x2 quad of the image: reads the three colour planes once, writes Y at full size and each chroma
// plane at its own reduction.  C `/` throughout (truncation towards zero: the chroma samples are signed).
static __device__ __forceinline__ void yk_reduce_quad(int a, int b, int c, int d, int hx, int hy, int mode,
                                                      int32_t* __restrict__ out, int ow, int qx, int qy) {
    // a b / c d = the quad at (2qx, 2qy); EDownSample (framework.h:60-66): 0 NEAREST_TL 1 NEAREST_BR 2 AVERAGE_BOX 3 MAX_BOX 4 MIN_BOX
    if (hx && hy) {
        int v = a;
        if (mode == 2) v = (a + b + c + d) / 4;
        else if (mode == 1) v = d;
        else if (mode == 3) v = max(max(a, b), max(c, d));
        else if (mode == 4) v = min(min(a, b), min(c, d));
        out[(size_t)qy * ow + qx] = v;
    } else if (hx) {                          // modes 0 and 2 only (the API refuses the others on one axis)
        out[(size_t)(2 * qy) * ow + qx] = mode == 2 ? (a + b) / 2 : a;
        out[(size_t)(2 * qy + 1) * ow + qx] = mode == 2 ? (c + d) / 2 : c;
    } else if (hy) {
        *reinterpret_cast<int2*>(out + (size_t)qy * ow + 2 * qx) = mode == 2 ? make_int2((a + c) / 2, (b + d) / 2) : make_int2(a, b);
    } else {
        *reinterpret_cast<int2*>(out + (size_t)(2 * qy) * ow + 2 * qx) = make_int2(a, b);
        *reinterpret_cast<int2*>(out + (size_t)(2 * qy + 1) * ow + 2 * qx) = make_int2(c, d);
    }
}

__global__ void __launch_bounds__(256)
yk_k_chroma(const YkSlotDev* __restrict__ slots, int slot, const YkChromaArgs A) {
    const YkSlotDev& S = slots[slot];
    const int qw = S.w >> 1, qh = S.h >> 1;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= qw * qh) return;
    const int qx = q % qw, qy = q / qw;
    int Y[4], Co[4], Cg[4];
#pragma unroll
    for (int row = 0; row < 2; row++) {
        const size_t at = (size_t)(2 * qy + row) * S.w + 2 * qx;
        const int2 R = __ldg(reinterpret_cast<const int2*>(S.plane[0] + at));
        const int2 G = __ldg(reinterpret_cast<const int2*>(S.plane[1] + at));
        const int2 B = __ldg(reinterpret_cast<const int2*>(S.plane[2] + at));
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const int r = k ? R.y : R.x, g = k ? G.y : G.x, b = k ? B.y : B.x;
            const int co = r - b, tmp = b + co / 2, cg = g - tmp;             // EC.cpp:55-66
            Y[2 * row + k] = tmp + cg / 2; Co[2 * row + k] = co / 2; Cg[2 * row + k] = cg / 2;
        }
    }
    *reinterpret_cast<int2*>(A.y + (size_t)(2 * qy) * S.w + 2 * qx) = make_int2(Y[0], Y[1]);
    *reinterpret_cast<int2*>(A.y + (size_t)(2 * qy + 1) * S.w + 2 * qx) = make_int2(Y[2], Y[3]);
    yk_reduce_quad(Co[0], Co[1], Co[2], Co[3], A.half[0], A.half[1], A.mode[0], A.co, A.half[0] ? qw : S.w, qx, qy);
    yk_reduce_quad(Cg[0], Cg[1], Cg[2], Cg[3], A.half[2], A.half[3], A.mode[1], A.cg, A.half[2] ? qw : S.w, qx, qy);
}

// ------------------------------------------------------------------------------------------------------------------// launch wrappers
void yk_launch_state(const YkSlotDev* slotsDev, int slot, int nRegions, int32_t* smoothMap, int32_t* mipmapMask,
                     int32_t* mappedRGB, int32_t* recon0, int32_t* recon1, int32_t* recon2, cudaStream_t st) {
    YK_LAUNCH(yk_k_state, dim3(nRegions), dim3(YK_THREADS), 0, st, slotsDev, slot, smoothMap, mipmapMask, mappedRGB, recon0, recon1, recon2);
}
void yk_launch_range_dyn_encode(const YkSlotDev* slotsDev, int slot, const YkR1Launch& launch, int numSMs, const int* lutDev, const uint16_t* rtabDev, const int16_t* r7Dev, cudaStream_t st) {
    const int maxBlocks = launch.walk.nBlocks;
    const int units = (maxBlocks + YK_R1_UNIT - 1) / YK_R1_UNIT;
    YK_LAUNCH(yk_k_r1_offsets, dim3(units > 0 ? units : 1), dim3(YK_R1_UNIT), 0, st, slotsDev, slot, launch);
    // warps take listed blocks with a grid stride: enough CTAs to fill every SM, no more than there can be blocks
    const bool three = launch.nJobs == 3;
    const int perCta = YK_R1_THREADS / 32;
    long long want = ((long long)maxBlocks + perCta - 1) / perCta;
    const long long cap = (long long)numSMs * (three ? YK_R1_CAP3 : YK_R1_CAP);
    if (want > cap) want = cap;
    const dim3 grid(want > 0 ? (unsigned)want : 1u);
    const unsigned short* rtab = reinterpret_cast<const unsigned short*>(rtabDev);
    const short* r7tab = reinterpret_cast<const short*>(r7Dev);
    if (three) {
        YK_LAUNCH(yk_k_r1_encode3, grid, dim3(YK_R1_THREADS), 0, st, slotsDev, slot, launch, lutDev, rtab, r7tab);
    } else {
        YK_LAUNCH(yk_k_r1_encode, grid, dim3(YK_R1_THREADS), 0, st, slotsDev, slot, launch, lutDev, rtab, r7tab);
    }
}
void yk_launch_chroma(const YkSlotDev* slotsDev, int slot, int w, int h, const YkChromaArgs& args, cudaStream_t st) {
    const int quads = (w >> 1) * (h >> 1);
    YK_LAUNCH(yk_k_chroma, dim3((quads + 255) / 256), dim3(256), 0, st, slotsDev, slot, args);
}

// CUDA loads kernels lazily, and loading one synchronises the context: a kernel that waits for another stream (yk_strip_run)
// would then never be released by a kernel that is launched for the first time.  Every kernel is loaded up front.
int yk_preload_aux() {
#ifndef YK_EMULATE
    cudaFuncAttributes fa;
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_state); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_r1_offsets); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_r1_encode); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_r1_encode3); if (e != cudaSuccess) return (int)e; }
    { const cudaError_t e = cudaFuncGetAttributes(&fa, yk_k_chroma); if (e != cudaSuccess) return (int)e; }
#endif
    return 0;
}
