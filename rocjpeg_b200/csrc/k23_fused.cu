// k23_fused.cu — dequantise + islow IDCT + chroma upsampling + colour conversion in ONE kernel (K2 + K3 fused), sm_100a.
//
// For ROCJPEG_OUTPUT_RGB / RGB_PLANAR of a whole picture the decoded component planes are an intermediate nobody asks
// for: K2 writes them to HBM only for K3 to read them back (a quarter of both kernels' traffic on the 500x375 batch).
// Here a CTA owns one MCU row of a 256-pixel-wide strip of one picture: it expands and transforms the strip's blocks
// (the VCN stage of the reference, src/rocjpeg_vaapi_decoder.cpp:677-689) into shared-memory planes and converts them
// to the caller's pixels right there (the reference's ColorConvertToRGB[Planar] kernels, src/rocjpeg_decoder.cpp:450-557,
// src/rocjpeg_hip_kernels.cpp:52-2029). Algorithmic bytes = coefficient entries + block records read, pixels written.
// The arithmetic is the two stages' own: idct_core.cuh and k3_rows.cuh, bit-exact with the un-fused path (which keeps
// serving crops, the planar formats the IDCT stage writes directly, the interleaved NATIVE surfaces and the test taps).
#include <cuda_runtime.h>

#include "idct_core.cuh"
#include "k3_rows.cuh"
#include "stages.h"

namespace rjb {
namespace {

using namespace idct;
using namespace k3;

constexpr int kStripW = 256;          // luma samples per strip (= kK3TileW: the row routines cover it with 8 per lane)
constexpr int kFThreads = 256;        // 32 blocks x 8 threads per IDCT batch; 8 warps for the rows
constexpr int kMaxBlocks = 128;       // blocks of one strip: 32 MCUs x 4 (4:4:0) or 16 MCUs x 8 ((2x2, 1x2, 1x2) 4:2:2)
constexpr int kLumaBytes = 16 * kStripW, kChromaBytes = 8 * kStripW;   // plane capacities: 16 rows of luma; 8 x 256 or 16 x 128 of chroma
static_assert(kStripW == kTileW, "the row routines assume 8 samples per lane over the strip");

__global__ void __launch_bounds__(kFThreads, 6) k23_fused(K23Args a) {
    PdlEntry();
    __shared__ __align__(16) int ws[32 * kBS];
    __shared__ __align__(16) uint8_t s_pl[kLumaBytes + 2 * kChromaBytes];
    __shared__ __align__(16) uint8_t s_buf[kFThreads / 32][kRowBuf];
    __shared__ uint32_t s_tab[3][64];            // per component and zig-zag code: TabEntry
    // per block of the strip: {first entry, entries | component << 16 | valid << 24, dequantised DC, plane offset | pitch << 16}
    __shared__ __align__(16) uint4 s_meta[kMaxBlocks];
    __shared__ K3Job s_job;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // every thread reads the picture's record itself (uniform loads, one cache line): no thread-0 prologue
    const FusedImage& fi = a.fused[__ldg(a.tile_img + blockIdx.x) & 0xFFFFu];
    const uint32_t t = blockIdx.x - fi.tile0;
    const int mrow = int(t / fi.tiles_x), tx = int(t - uint32_t(mrow) * fi.tiles_x);
    const int m0 = tx * fi.mpt, nm = min(fi.mpt, fi.mcus_x - m0);
    const int ncomp = fi.ncomp;
    const int nbw0 = nm * fi.H[0], nbw1 = ncomp > 1 ? nm * fi.H[1] : 0, nbw2 = ncomp > 2 ? nm * fi.H[2] : 0;
    const int cnt0 = nbw0 * fi.V[0], cnt1 = nbw1 * (ncomp > 1 ? fi.V[1] : 0), cnt2 = nbw2 * (ncomp > 2 ? fi.V[2] : 0);
    const int nblocks = cnt0 + cnt1 + cnt2;
    const uint32_t* entries = a.entries + fi.ent0;
    const BlockRec* rec = a.blk_rec + fi.blk0;
    const int xt = tx * kStripW, rows = 8 * fi.vmax, y0t = mrow * rows;
    if (tid == 0) {
        // the row routines see the strip's shared-memory planes through pointers whose origin is the picture's (0, 0)
        K3Job j;
        for (int c = 0; c < 3; c++) {
            const int cc = c < ncomp ? c : 0;
            const int shx = cc ? fi.sx : 0, shy = cc ? fi.sy : 0;
            j.pitch[c] = fi.pitch[cc];
            j.p[c] = s_pl + fi.base[cc] - (size_t(y0t >> shy) * fi.pitch[cc] + size_t(xt >> shx));
            j.dst[c] = fi.dst[c];
            j.dpitch[c] = fi.dpitch;
        }
        j.dst[3] = nullptr;
        j.dpitch[3] = 0;
        j.W = fi.width; j.H = fi.height; j.x0 = 0; j.y0 = 0; j.css = fi.css; j.fmt = fi.fmt;
        j.xt = xt;
        j.ty = mrow;
        j.nx = min(kStripW, fi.width - xt);
        s_job = j;
    }
    // quantiser / offset tables per component
    for (int idx = tid; idx < ncomp * 64; idx += kFThreads) {
        const int c = idx >> 6, code = idx & 63;
        s_tab[c][code] = TabEntry(code, a.qtables + size_t(fi.qidx[c]) * 64);
    }
    // per block of the strip: its record (where its entries lie, integrated DC) and where its samples go
    if (tid < kMaxBlocks) {
        uint4 m = make_uint4(0u, 0u, 0u, 0u);
        if (tid < nblocks) {
            int g = tid, c = 0, nbw = nbw0;
            if (g >= cnt0) { g -= cnt0; c = 1; nbw = nbw1; if (g >= cnt1) { g -= cnt1; c = 2; nbw = nbw2; } }
            const int v = g / nbw, bx = g - v * nbw;
            const int H = fi.H[c];
            const size_t blk = size_t(mrow * fi.mcus_x + m0 + (bx >> fi.hshift[c])) * size_t(fi.bpm) + size_t(fi.first_blk[c] + v * H + (bx & (H - 1)));
            const uint2 r = __ldg(reinterpret_cast<const uint2*>(rec + blk));
            const uint2 e = BlockEntryRange(blk ? __ldg(&rec[blk - 1].end) : 0u, r.x, fi.ent_cap);
            m.x = e.x;
            m.y = (e.y - e.x) | (uint32_t(c) << 16) | (1u << 24);
            m.z = uint32_t(int(int16_t(r.y & 0xFFFFu)) * int(__ldg(a.qtables + size_t(fi.qidx[c]) * 64)));   // integrated DC, dequantised
            m.w = (fi.base[c] + uint32_t(v * 8) * fi.pitch[c] + uint32_t(bx * 8)) | (fi.pitch[c] << 16);
        }
        s_meta[tid] = m;
    }
    __syncthreads();
    // ---- IDCT: 32 blocks at a time, 8 threads per block, samples to shared memory. The loop is issue bound: everything it
    // touches is addressed through 32-bit shared-window addresses computed once, a block's description is one 128-bit load,
    // and the trip count is the same for every warp.
    const int b = tid >> 3, jj = tid & 7;
    const uint32_t my_sa = SharedU32(ws) + uint32_t(b * kBS * 4);
    const uint32_t row_sa = my_sa + uint32_t(jj * kRS * 4), col_sa = my_sa + uint32_t(jj * 4);
    const uint32_t tab_sa0 = SharedU32(&s_tab[0][0]), pl_sa = SharedU32(s_pl);
    uint32_t meta_sa = SharedU32(s_meta) + uint32_t(b * 16);
    const uint32_t* const ent_j = entries + jj;
    const uint32_t meta_end = SharedU32(s_meta) + uint32_t(nblocks * 16);
#pragma unroll 1
    for (; meta_sa < meta_end + uint32_t(b * 16); meta_sa += 32 * 16) {   // (same trip count for the 32 block slots: slot b's g runs b, b + 32, ...)
        const uint4 m = Lds128(meta_sa);
        ScatterColumns(my_sa, row_sa, col_sa, jj, tab_sa0, (m.y >> 8) & 0x300u, ent_j + m.x, m.y & 0xFFFFu, m.z);
        int out[8];
        RowPass(row_sa, out);
        if (m.y >> 24) Sts64(pl_sa + (m.w & 0xFFFFu) + uint32_t(jj) * (m.w >> 16), PackRow(out));
        __syncwarp();
    }
    __syncthreads();
    // ---- rows: upsample + convert + store (k3_output.cu's RGB rows, planes in shared memory) ----
    const K3Job& j = s_job;
    const int fmt = j.fmt, css = j.css;
    if (j.nx <= 0) return;
    if (fmt == FMT_RGB && (j.dst[0] == nullptr || j.dpitch[0] == 0)) return;
    if (fmt == FMT_RGB_PLANAR && (!j.dst[0] || !j.dst[1] || !j.dst[2] || j.dpitch[0] == 0)) return;
    const int sx = css == CSS_411 ? 2 : (css == CSS_422 || css == CSS_420) ? 1 : 0;
    const int sy = (css == CSS_440 || css == CSS_420) ? 1 : 0;
    const bool gray = (css == CSS_400);
    const uintptr_t bases = fmt == FMT_RGB ? reinterpret_cast<uintptr_t>(j.dst[0]) + size_t(j.xt) * 3
                                           : (reinterpret_cast<uintptr_t>(j.dst[0]) | reinterpret_cast<uintptr_t>(j.dst[1]) |
                                              reinterpret_cast<uintptr_t>(j.dst[2])) + size_t(j.xt);
    uint8_t* buf = s_buf[warp];
    for (int r = warp; r < rows; r += kFThreads / 32) {
        const int y = y0t + r;
        if (y >= j.H) break;
        const bool dst_ok = ((bases | (size_t(y) * j.dpitch[0])) & 3) == 0;
        if (dst_ok) {
            if (sx == 2) RowRgbFast<2, true>(j, sy, gray, y, lane); else if (sx) RowRgbFast<1, true>(j, sy, gray, y, lane); else RowRgbFast<0, true>(j, sy, gray, y, lane);
        } else {
            if (sx == 2) RowRgbStaged<2, true>(j, sy, gray, buf, y, lane); else if (sx) RowRgbStaged<1, true>(j, sy, gray, buf, y, lane);
            else RowRgbStaged<0, true>(j, sy, gray, buf, y, lane);
        }
    }
}


// ---------------------------------------------------------------- k23_warp: the same work, one warp per 32-sample column
//
// Pictures whose destination rows are all 4-byte aligned (base and pitch multiples of 4: every row takes the register
// path) need no CTA-wide staging, so nothing has to be shared between the warps of a CTA but the quantiser tables: each
// warp owns the MCUs under 32 luma samples of the strip - 4, 2 or 1 of them, at most 16 blocks - transforms them into
// its own planes (1 KiB) and converts those rows itself, eight 32-pixel row segments per pass. No barrier after the
// table set-up: a warp waiting for its records or entries no longer holds seven others at a CTA barrier (a sixth of the
// strip kernel's stall samples, profiles/r02z_c3_hot.md).
constexpr int kWarpW = 32;                 // luma samples per warp
constexpr int kWarpBlocks = 16;            // blocks under them at most ((2x2, 1x2, 1x2) and 4:4:0: 16; 4:4:4 and 4:2:0: 12)
constexpr int kWarpLuma = kWarpW * 16, kWarpChroma = 256;   // plane capacities: 32 x 16 luma; 32 x 8, 16 x 16 or 8 x 8 chroma

struct __align__(16) WarpSmem {
    int ws[4 * kBS];                       // four blocks in flight
    uint4 meta[kWarpBlocks];
    uint8_t pl[kWarpLuma + 2 * kWarpChroma];
};

__global__ void __launch_bounds__(kFThreads, 6) k23_warp(K23Args a) {
    PdlEntry();
    __shared__ WarpSmem s_w[kFThreads / 32];
    __shared__ uint32_t s_tab[3][64];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = __ldg(a.tile_img_w + blockIdx.x);
    const FusedImage& gfi = a.fused[tile & 0xFFFFu];
    // the picture's record into shared memory: every warp reads a dozen of its fields, each a dependent global load otherwise
    // (a quarter of the kernel's stall samples sat in the per-warp set-up, profiles/r03z_c3_hot.md)
    __shared__ __align__(16) FusedImage s_fi;
    static_assert(sizeof(FusedImage) % 16 == 0, "copied as 16-byte vectors");
    if (tid < int(sizeof(FusedImage) / 16)) reinterpret_cast<uint4*>(&s_fi)[tid] = __ldg(reinterpret_cast<const uint4*>(&gfi) + tid);
    {
        const int ncomp_g = gfi.ncomp;
        for (int idx = tid; idx < ncomp_g * 64; idx += kFThreads) {
            const int c = idx >> 6, code = idx & 63;
            s_tab[c][code] = TabEntry(code, a.qtables + size_t(gfi.qidx[c]) * 64);
        }
    }
    __syncthreads();
    const FusedImage& fi = s_fi;
    const int mrow = int(tile >> 16), tx = int(blockIdx.x - fi.tile0) - mrow * int(fi.tiles_x);
    const int ncomp = fi.ncomp;
    const int mpt = fi.mpt, mcus_x = fi.mcus_x;
    const int mpw = mpt >> 3;                          // MCUs per warp: 4 (8-sample MCUs), 2 or 1
    const int m0 = tx * mpt + warp * mpw, nm = min(mpw, mcus_x - m0);
    if (nm <= 0) return;
    WarpSmem& sw = s_w[warp];
    // ---- the warp's blocks: record, dequantised DC, where the samples go (V <= 2: no division anywhere)
    int nblocks;
    {
        const uint32_t ci0 = fi.comp_info[0], ci1 = ncomp > 1 ? fi.comp_info[1] : 0u, ci2 = ncomp > 2 ? fi.comp_info[2] : 0u;
        const int nbw0 = nm * int(ci0 & 0xFFu), nbw1 = nm * int(ci1 & 0xFFu), nbw2 = nm * int(ci2 & 0xFFu);
        const int cnt0 = nbw0 * int((ci0 >> 8) & 0xFFu), cnt1 = nbw1 * int((ci1 >> 8) & 0xFFu), cnt2 = nbw2 * int((ci2 >> 8) & 0xFFu);
        nblocks = cnt0 + cnt1 + cnt2;
        if (lane < kWarpBlocks) {
            uint4 m = make_uint4(0u, 0u, 0u, 0u);
            if (lane < nblocks) {
                int g = lane, c = 0, nbw = nbw0;
                uint32_t ci = ci0;
                if (g >= cnt0) { g -= cnt0; c = 1; nbw = nbw1; ci = ci1; if (g >= cnt1) { g -= cnt1; c = 2; nbw = nbw2; ci = ci2; } }
                const int v = g >= nbw ? 1 : 0, bx = g - (v ? nbw : 0);
                const uint32_t H = ci & 0xFFu;
                const uint32_t blk = uint32_t(mrow * mcus_x + m0 + (bx >> (ci >> 24))) * uint32_t(fi.bpm) + ((ci >> 16) & 0xFFu) + uint32_t(v) * H + (uint32_t(bx) & (H - 1u));
                const BlockRec* rp = a.blk_rec + fi.blk0 + blk;
                const uint2 r = __ldg(reinterpret_cast<const uint2*>(rp));
                const uint2 e = BlockEntryRange(blk ? __ldg(&rp[-1].end) : 0u, r.x, fi.ent_cap);
                const uint32_t pitch = uint32_t(8 * mpw) * H;                       // 32 for luma, 32 >> sx for chroma
                const uint32_t base = c == 0 ? 0u : uint32_t(kWarpLuma + (c - 1) * kWarpChroma);
                m.x = e.x;
                m.y = (e.y - e.x) | (uint32_t(c) << 16) | (1u << 24);
                m.z = uint32_t(int(int16_t(r.y & 0xFFFFu)) * int(s_tab[c][1] >> 16));   // integrated DC, dequantised (code 1 = position 0)
                m.w = (base + uint32_t(v * 8) * pitch + uint32_t(bx * 8)) | (pitch << 16);
            }
            sw.meta[lane] = m;
        }
    }
    __syncwarp();
    // ---- IDCT, four blocks per step (the strip kernel's loop)
    {
        const int b = lane >> 3, jj = lane & 7;
        const uint32_t my_sa = SharedU32(sw.ws) + uint32_t(b * kBS * 4);
        const uint32_t row_sa = my_sa + uint32_t(jj * kRS * 4), col_sa = my_sa + uint32_t(jj * 4);
        const uint32_t tab_sa0 = SharedU32(&s_tab[0][0]), pl_sa = SharedU32(sw.pl);
        uint32_t meta_sa = SharedU32(sw.meta) + uint32_t(b * 16);
        const uint32_t* const ent_j = a.entries + fi.ent0 + jj;
        const uint32_t meta_end = meta_sa + uint32_t(nblocks * 16);
#pragma unroll 1
        for (; meta_sa < meta_end; meta_sa += 4 * 16) {
            const uint4 m = Lds128(meta_sa);
            ScatterColumns(my_sa, row_sa, col_sa, jj, tab_sa0, (m.y >> 8) & 0x300u, ent_j + m.x, m.y & 0xFFFFu, m.z);
            int out[8];
            RowPass(row_sa, out);
            if (m.y >> 24) Sts64(pl_sa + (m.w & 0xFFFFu) + uint32_t(jj) * (m.w >> 16), PackRow(out));
            __syncwarp();
        }
    }
    // ---- rows: eight 32-pixel segments per pass, 8 pixels per lane
    const int fmt = fi.fmt;
    uint8_t* const d0 = fi.dst[0];
    uint8_t* const d1 = fi.dst[1];
    uint8_t* const d2 = fi.dst[2];
    const uint32_t dpitch = fi.dpitch;
    if (d0 == nullptr || dpitch == 0) return;
    if (fmt == FMT_RGB_PLANAR && (!d1 || !d2)) return;
    const bool gray = fi.css == CSS_400;
    const int sx = fi.sx, sy = fi.sy;
    const int rows = 8 * fi.vmax, y0 = mrow * rows;
    const int seg = lane & 3, x = tx * kStripW + warp * kWarpW + seg * 8;
    const int n = fi.width - x;
    if (n <= 0) return;
    const uint32_t pl_sa = SharedU32(sw.pl);
    const uint32_t cp = ncomp > 1 ? uint32_t(8 * mpw * fi.H[1]) : 0u;   // chroma pitch (32 >> sx for the usual sampling factors)
    for (int r = lane >> 2; r < rows; r += 8) {
        const int y = y0 + r;
        if (y >= fi.height) break;
        uint2 yy;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(yy.x), "=r"(yy.y) : "r"(pl_sa + uint32_t(r * kWarpW + seg * 8)));
        Rgb8 o;
        if (gray) {
            o.r = o.g = o.b = yy;
        } else {
            const uint32_t ca = pl_sa + uint32_t(kWarpLuma) + uint32_t(r >> sy) * cp + uint32_t((seg * 8) >> sx);
            uint2 uu = make_uint2(0u, 0u), vv = make_uint2(0u, 0u);
            if (sx == 0) {
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(uu.x), "=r"(uu.y) : "r"(ca));
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(vv.x), "=r"(vv.y) : "r"(ca + uint32_t(kWarpChroma)));
                o = Convert8<0>(yy, uu, vv);
            } else if (sx == 1) {
                uu.x = Lds32(ca);
                vv.x = Lds32(ca + uint32_t(kWarpChroma));
                o = Convert8<1>(yy, uu, vv);
            } else {
                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(uu.x) : "r"(ca));
                asm volatile("ld.shared.u16 %0, [%1];" : "=r"(vv.x) : "r"(ca + uint32_t(kWarpChroma)));
                o = Convert8<2>(yy, uu, vv);
            }
        }
        StoreRgb8(fmt, d0, d1, d2, dpitch, y, x, n, o);
    }
}

}  // namespace

cudaError_t LaunchK23Fused(const K23Args& a, cudaStream_t stream, uint32_t* launches) {
    cudaError_t e = cudaSuccess;
    if (a.total_tiles_w != 0) e = LaunchPdl(launches, k23_warp, dim3(a.total_tiles_w), dim3(kFThreads), 0, stream, a);
    if (e == cudaSuccess && a.total_tiles != 0) e = LaunchPdl(launches, k23_fused, dim3(a.total_tiles), dim3(kFThreads), 0, stream, a);
    return e;
}

cudaError_t PreloadK23() {
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, k23_fused);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k23_warp);
    return e;
}

}  // namespace rjb
