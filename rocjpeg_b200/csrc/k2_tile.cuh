// k2_tile.cuh — what the IDCT kernels share: the tile -> picture / component resolution and the records of a
// tile's blocks. The full-size kernel (k2_idct.cu) and the reduced-size kernels (k2_scaled.cu) cut a component
// into the same tiles: 32 horizontally adjacent blocks of one block row. They differ in how many samples a block
// yields per row and column: S = 8 at full size, 8 / d at scale 1/d.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "idct_core.cuh"
#include "stages.h"

namespace rjb {
namespace k2tile {

constexpr int kBlocksPerTile = 32;
constexpr int kSearchCache = 1024;   // image tile prefix entries searched in shared memory

// Everything the threads of a CTA need about one tile (32 adjacent blocks of one block row
// of one component), resolved once per tile by one thread.
struct TileInfo {
    const uint32_t* entries; // image's coefficient entries
    const BlockRec* rec;     // image's per-block records (a block's entries begin where its predecessor's end)
    uint32_t ent_cap;
    const uint16_t* qt;      // natural-order quantiser table of the component
    uint8_t* out;            // plane address of (row by*S, column 0)
    uint32_t pitch;
    uint32_t row_mcu;        // (by / V) * mcus_x
    uint32_t k_row;          // comp_first_blk + (by % V) * H
    int32_t bx0, nbx;        // first block column of the tile, block columns of the component (<0: no more tiles)
    int32_t hshift, hmask, bpm;
    // direct mode (planar output formats without a crop): `out`/`pitch` address the caller's channel,
    // stores are clipped to the component's visible size and follow the destination's alignment
    int32_t direct;          // 0: plane arena; 1: caller's buffer; 2: nothing to store (channel skipped / not part of the format)
    int32_t clip_w, clip_rows;
};

// largest i in [0, n) with a[i] <= v; the prefix array is searched in its shared-memory copy when it
// fits (eight dependent global loads per tile were a fifth of the kernel: profiles/r01f_*)
__device__ __forceinline__ uint32_t UpperIndexK2(const uint32_t* a, const uint32_t* cached, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    if (cached) {
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (cached[mid] <= v) lo = mid; else hi = mid;
        }
    } else {
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
        }
    }
    return lo;
}

// picture size at scale 1/D: ceil(n / D) (libjpeg's output_width / output_height for scale_denom D)
template <int D>
__device__ __forceinline__ int Scaled(int n) { return D == 1 ? n : (n + D - 1) / D; }

// tile -> (image, component, block row, first block column); sampling factors are powers of two,
// so no division in the hot part. S = samples per block row and column (8 / scale denominator): the
// picture's output is ceil(width * S / 8) x ceil(height * S / 8) luma samples, the crop rectangle and
// the caller's channels are in those units.
template <int S>
__device__ __forceinline__ TileInfo ResolveTile(const K2Args& a, const uint32_t* cached_tile0, uint32_t tile) {
    constexpr int kLogS = S == 8 ? 3 : S == 4 ? 2 : S == 2 ? 1 : 0;
    constexpr int kDen = 8 / S;
    TileInfo ti = {};
    ti.nbx = -1;
    if (tile >= a.total_tiles) return ti;
    const uint32_t img = UpperIndexK2(a.img_tile0, cached_tile0, uint32_t(a.nimages), tile);
    const ImageDesc& im = a.images[img];
    uint32_t t = tile - a.img_tile0[img];
    for (int comp = 0; comp < im.ncomp; comp++) {
        const uint32_t tiles_x = (uint32_t(im.blocks_w[comp]) + kBlocksPerTile - 1) / kBlocksPerTile;
        const uint32_t n = tiles_x * uint32_t(im.blocks_h[comp]);
        if (t < n) {
            const int by = int(t / tiles_x);
            const int H = im.hs[comp], V = im.vs[comp];
            const int hs = __ffs(H) - 1, vs = __ffs(V) - 1;
            ti.entries = a.entries + im.ent0;
            ti.rec = a.blk_rec + im.blk0;
            ti.ent_cap = im.ent_cap;
            ti.qt = a.qtables + size_t(im.qt_index[comp]) * 64;
            ti.pitch = im.plane_pitch[comp];
            ti.out = a.planes + im.plane_off[comp] + size_t(by) * S * ti.pitch;
            ti.row_mcu = uint32_t(by >> vs) * uint32_t(im.mcus_x);
            ti.k_row = uint32_t(im.comp_first_blk[comp] + ((by & (V - 1)) << hs));
            ti.bx0 = int(t % tiles_x) * kBlocksPerTile;
            ti.nbx = im.blocks_w[comp];
            ti.hshift = hs;
            ti.hmask = H - 1;
            ti.bpm = im.bpm;
            const OutputDesc& od = a.outputs[img];
            if (od.fused && !a.force_planes) ti.direct = 2;   // the fused kernel transforms this picture's blocks itself
            if (!od.direct && !a.force_planes && (od.x0 != 0 || od.y0 != 0 || od.w != Scaled<kDen>(im.width) || od.h != Scaled<kDen>(im.height))) {
                // Region of interest (src/rocjpeg_decoder.cpp:120-141): the output stage only reads the
                // samples under the crop rectangle, so blocks outside it are not transformed at all.
                const int sx = comp == 0 ? 0 : im.css == CSS_411 ? 2 : (im.css == CSS_422 || im.css == CSS_420) ? 1 : 0;
                const int sy = (comp != 0 && (im.css == CSS_440 || im.css == CSS_420)) ? 1 : 0;
                int x_lo = od.x0, x_hi = od.x0 + od.w - 1, y_lo = od.y0, y_hi = od.y0 + od.h - 1;
                if (od.jfif) {
                    // fancy upsampling (k3_jfif.cu) reads one chroma sample beyond the crop on each side: the rectangle
                    // widened by one chroma sample, clamped to the picture
                    const int hx = im.css == CSS_411 ? 4 : (im.css == CSS_422 || im.css == CSS_420) ? 2 : 1;
                    const int hy = (im.css == CSS_440 || im.css == CSS_420) ? 2 : 1;
                    x_lo = max(0, x_lo - hx); x_hi = min(od.pic_w - 1, x_hi + hx);
                    y_lo = max(0, y_lo - hy); y_hi = min(od.pic_h - 1, y_hi + hy);
                }
                const int bx_lo = (x_lo >> sx) >> kLogS, bx_hi = (x_hi >> sx) >> kLogS;
                const int by_lo = (y_lo >> sy) >> kLogS, by_hi = (y_hi >> sy) >> kLogS;
                if (by < by_lo || by > by_hi || ti.bx0 > bx_hi || ti.bx0 + kBlocksPerTile - 1 < bx_lo) ti.direct = 2;
            }
            if (od.direct && !a.force_planes) {
                // channel, pitch and visible size of this component in the caller's layout
                // (src/rocjpeg_decoder.cpp:576-636: planar chroma at the subsampled size, floor shifts;
                // 4:2:2 / 4:2:0 use pitch[1] for both chroma planes, 4:4:4 / 4:4:0 each channel's own)
                const int sx = im.css == CSS_411 ? 2 : (im.css == CSS_422 || im.css == CSS_420) ? 1 : 0;
                const int sy = (im.css == CSS_440 || im.css == CSS_420) ? 1 : 0;
                const uint32_t dpitch = comp == 0 ? od.dst_pitch[0] : (sx == 0 ? od.dst_pitch[comp] : od.dst_pitch[1]);
                const int cw = comp == 0 ? Scaled<kDen>(im.width) : (Scaled<kDen>(im.width) >> sx),
                          chh = comp == 0 ? Scaled<kDen>(im.height) : (Scaled<kDen>(im.height) >> sy);
                const bool wanted = comp == 0 || od.fmt != FMT_Y;
                if (!wanted || od.dst[comp] == nullptr || dpitch == 0 || by * S >= chh) {
                    ti.direct = 2;
                } else {
                    ti.direct = 1;
                    ti.pitch = dpitch;
                    ti.out = od.dst[comp] + size_t(by) * S * dpitch;
                    ti.clip_w = cw;
                    ti.clip_rows = min(S, chh - by * S);
                }
            }
            break;
        }
        t -= n;
    }
    return ti;
}

// The CTA's kTiles tiles, resolved into s_tile by its first kTiles threads (the image tile prefix searched in s_tile0
// when it fits there); ends with the CTA synchronised.
template <int S, int kThreads, int kTiles>
__device__ __forceinline__ void ResolveCtaTiles(const K2Args& a, TileInfo* s_tile, uint32_t* s_tile0) {
    const int tid = threadIdx.x;
    const bool cached = a.nimages <= kSearchCache;
    if (cached) {
        for (int i = tid; i < a.nimages; i += kThreads) s_tile0[i] = __ldg(a.img_tile0 + i);
        __syncthreads();
    }
    if (tid < kTiles) s_tile[tid] = ResolveTile<S>(a, cached ? s_tile0 : nullptr, blockIdx.x * kTiles + tid);
    __syncthreads();
}

// decode-order index of the tile's block in block column bx
__device__ __forceinline__ size_t TileBlock(const TileInfo& ti, int bx) {
    return size_t(ti.row_mcu + uint32_t(bx >> ti.hshift)) * uint32_t(ti.bpm) + ti.k_row + uint32_t(bx & ti.hmask);
}

// Block bb of the tile for the transform loops: {first entry, entries | valid << 24, dequantised integrated DC, 0}; zero
// past the component's right edge and in a tile with nothing to store
__device__ __forceinline__ uint4 TileBlockMeta(const TileInfo& ti, int bb) {
    uint4 m = make_uint4(0u, 0u, 0u, 0u);
    if (ti.nbx >= 0 && ti.direct != 2 && ti.bx0 + bb < ti.nbx) {
        const size_t blk = TileBlock(ti, ti.bx0 + bb);
        const uint2 r = __ldg(reinterpret_cast<const uint2*>(ti.rec + blk));
        const uint2 e = BlockEntryRange(blk ? __ldg(&ti.rec[blk - 1].end) : 0u, r.x, ti.ent_cap);
        m.x = e.x;
        m.y = (e.y - e.x) | (1u << 24);
        m.z = uint32_t(int(int16_t(r.y & 0xFFFFu)) * int(__ldg(ti.qt)));   // integrated DC, dequantised
    }
    return m;
}

}  // namespace k2tile
}  // namespace rjb
