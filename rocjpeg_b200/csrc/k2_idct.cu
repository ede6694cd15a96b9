// k2_idct.cu — fused dequantise + integer "islow" 8x8 inverse DCT (K2) for sm_100a.
//
// Replaces the dequantisation + IDCT the reference delegates to the VCN
// fixed-function engine (src/rocjpeg_vaapi_decoder.cpp:677-689, 816-828). The
// arithmetic is libjpeg's jidctint.c islow (CONST_BITS 13, PASS1_BITS 2), which
// BASELINE.json mandates: column pass on coef*quant descaled by 11 bits, row pass
// descaled by 18 bits, +128, clamp — bit-exact with libjpeg-turbo's
// jpeg_idct_islow on encoder-produced data (the zero-column shortcuts in
// libjpeg are arithmetically identical to the general path, so none are taken).
//
// Input is K1's sparse coefficient stream: per block the index one past its last entry (it begins
// where the previous block of the image ends), one
// 32-bit (zig-zag position, int16 value) entry per non-zero coefficient, plus the integrated DC
// from the compact per-block array; the 8 threads of a block scatter the entries (dequantised)
// into a zeroed shared-memory workspace. Mapping: 8 threads per block, 32
// horizontally adjacent blocks of one component per tile, kTilesPerCta tiles per
// CTA, transposes through padded shared memory (bank-conflict free), one 8-byte
// store per thread = full 32-byte sectors per block row. The kernel was
// instruction-issue bound in its first form (profiles/r01a_c3_kernels.md), hence:
// no integer division (sampling factors are powers of two), rounding and the
// +128 level shift folded into the even part, cvt.pack.sat for the clamp+pack.
#include <cuda_runtime.h>

#include "idct_core.cuh"
#include "k2_tile.cuh"
#include "stages.h"

namespace rjb {
namespace {

using namespace idct;
using namespace k2tile;

constexpr int kThreads = kBlocksPerTile * 8;
constexpr int kTilesPerCta = 16;   // (8: a fifth of the warp time went to the barriers of the per-CTA set-up, profiles/r03l_*)

// 8 samples of one block row into the caller's buffer: n = visible samples left in the row
__device__ __forceinline__ void StoreClipped(uint8_t* dst, uint2 v, int n) {
    const uintptr_t al = reinterpret_cast<uintptr_t>(dst);
    if (n >= 8 && (al & 7) == 0) {
        *reinterpret_cast<uint2*>(dst) = v;
    } else if (n >= 8 && (al & 3) == 0) {
        reinterpret_cast<uint32_t*>(dst)[0] = v.x;
        reinterpret_cast<uint32_t*>(dst)[1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (i < n) dst[i] = uint8_t(((i < 4 ? v.x : v.y) >> (8 * (i & 3))) & 0xFFu);
    }
}

// 8 CTAs of 256 threads per SM (32 registers): the stage is latency/issue bound and lost 11% when a
// refactor let it grow to 40 registers. (A one-thread-per-block mapping — private shared-memory
// column, no transposes, ~30% fewer instructions — was measured 22-28% SLOWER: 77 registers and
// 33 KiB per CTA leave 24 warps per SM.)
__global__ void __launch_bounds__(kThreads, 8) k2_idct(K2Args a) {
    PdlEntry();
    // Workspace [block][row][col], row stride kRS = 12 words, block stride kBS = 104 words. A warp holds
    // 4 blocks x 8 threads: column-wise, thread (b, j) touches word 104 b + 12 r + j -> bank 8 b + j + const,
    // all 32 distinct; row-wise it moves its row as two 128-bit accesses whose bank groups 3 j mod 8 are
    // distinct within each quarter-warp.
    constexpr int kRS = 12, kBS = 104;
    __shared__ __align__(16) int ws[kBlocksPerTile * kBS];
    __shared__ TileInfo s_tile[kTilesPerCta];
    // per tile and zig-zag code of an entry: byte offset of the coefficient inside a block's workspace
    // (low half) and its quantiser step (high half) - one shared load replaces the zig-zag lookup, the
    // row/column split and the quantiser load
    __shared__ uint32_t s_tab[kTilesPerCta][64];
    __shared__ uint32_t s_tile0[kSearchCache];
    // per tile and block: {first entry, entries | valid << 24, dequantised integrated DC, -}
    __shared__ __align__(16) uint4 s_meta[kTilesPerCta][kBlocksPerTile];
    static_assert((kTilesPerCta * kBlocksPerTile) % kThreads == 0, "whole record fetches per thread");
    const int tid = threadIdx.x;
    const bool cached = a.nimages <= kSearchCache;
    if (cached) {
        for (int i = tid; i < a.nimages; i += kThreads) s_tile0[i] = __ldg(a.img_tile0 + i);
        __syncthreads();
    }
    if (tid < kTilesPerCta) s_tile[tid] = ResolveTile<8>(a, cached ? s_tile0 : nullptr, blockIdx.x * kTilesPerCta + tid);
    __syncthreads();
    for (int idx = tid; idx < kTilesPerCta * 64; idx += kThreads) {
        const int t = idx >> 6, code = idx & 63;   // entries carry position + 1 (huff_core.cuh)
        const TileInfo& ti = s_tile[t];
        if (ti.nbx >= 0) {
            const int nat = kZigzag[(code + 63) & 63];
            // (code 1 = position 0: DC-difference and pad entries - the integrated DC goes in with the zero fill - are parked in
            // a padding word of the workspace's first row)
            s_tab[t][code] = uint32_t(code == 1 ? 8 * 4 : ((nat >> 3) * kRS + (nat & 7)) * 4) | (uint32_t(__ldg(ti.qt + nat)) << 16);
        }
    }
    __syncthreads();
    const int b = tid >> 3, j = tid & 7;
    // Records of ALL the CTA's tiles first: every thread fetches the record pair of one (tile, block) -
    // eight tiles x 32 blocks = 256 - so the tile loop below starts from shared memory instead of
    // waiting for a dependent global load at the top of every tile (profiles/r01g_*).
#pragma unroll
    for (int rep = 0; rep < kTilesPerCta * kBlocksPerTile / kThreads; rep++) {
        const int t = (tid >> 5) + rep * (kThreads / 32), bb = tid & 31;
        const TileInfo& ti = s_tile[t];
        uint4 m = make_uint4(0u, 0u, 0u, 0u);
        if (ti.nbx >= 0 && ti.direct != 2 && ti.bx0 + bb < ti.nbx) {
            const int bx = ti.bx0 + bb;
            const size_t blk = size_t(ti.row_mcu + uint32_t(bx >> ti.hshift)) * uint32_t(ti.bpm) + ti.k_row + uint32_t(bx & ti.hmask);
            const uint2 r = __ldg(reinterpret_cast<const uint2*>(ti.rec + blk));
            uint32_t e0 = blk ? __ldg(&ti.rec[blk - 1].end) : 0u, e1 = r.x;
            // (a block of a valid stream has at most 64 entries + 7 pads per subsequence boundary inside it; after a DAMAGED
            // restart interval the first block of the next one also owns the pad groups the counting pass reserved in vain,
            // any number of them - they are skipped, not a reason to drop the block; the count is 16 bits wide)
            if (e0 == kNoEntry || e1 == kNoEntry || e1 < e0 || e1 - e0 > 0xFFFFu || e1 > ti.ent_cap) e1 = e0 = 0;   // never decoded
            m.x = e0;
            m.y = (e1 - e0) | (1u << 24);
            m.z = uint32_t(int(int16_t(r.y & 0xFFFFu)) * int(__ldg(ti.qt)));   // integrated DC, dequantised
        }
        s_meta[t][bb] = m;
    }
    __syncthreads();
    const uint32_t my_sa = SharedU32(ws) + uint32_t(b * kBS * 4);
    const uint32_t row_sa = my_sa + uint32_t(j * kRS * 4), col_sa = my_sa + uint32_t(j * 4);
    const uint32_t tab_sa0 = SharedU32(&s_tab[0][0]);
    const uint32_t meta_sa0 = SharedU32(&s_meta[0][0]) + uint32_t(b * 16);
#pragma unroll 1
    for (int it = 0; it < kTilesPerCta; it++) {
        const TileInfo& ti = s_tile[it];
        if (ti.nbx < 0) break;
        if (ti.direct == 2) continue;   // e.g. chroma of a colour picture decoded to ROCJPEG_OUTPUT_Y
        const uint4 m = Lds128(meta_sa0 + uint32_t(it * kBlocksPerTile * 16));
        const uint32_t n = m.y & 0xFFFFu;
        // expand the block's sparse entries into the zeroed workspace, dequantising on the way; four loads in flight
        // per thread (32 entries per block) before the first is used
        const uint32_t* ep = ti.entries + m.x + uint32_t(j);
        const uint32_t k = uint32_t(j);
        uint32_t e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) e[u] = (k + 8u * u < n) ? __ldg(ep + 8 * u) : 0u;
        Sts128(row_sa, make_uint4(j == 0 ? m.z : 0u, 0u, 0u, 0u));   // zero fill; the integrated DC goes in with it
        Sts128(row_sa + 16, make_uint4(0u, 0u, 0u, 0u));
        __syncwarp();
        const uint32_t tab_sa = tab_sa0 + uint32_t(it * 256);
        auto put = [&](uint32_t en) {
            const uint32_t t = Lds32(tab_sa + ((en >> 14) & 0xFCu));
            Sts32(my_sa + (t & 0xFFFFu), uint32_t(int(int16_t(en & 0xFFFFu)) * int(t >> 16)));
        };
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (k + 8u * u < n) put(e[u]);
        for (uint32_t kk = k + 32u; kk < n; kk += 8) put(__ldg(ep + (kk - k)));
        __syncwarp();
        int in[8], out[8];
#pragma unroll
        for (int r = 0; r < 8; r++) in[r] = int(Lds32(col_sa + uint32_t(r * kRS * 4)));   // column j
        Islow8<11>(in, out, 1 << 10);
#pragma unroll
        for (int r = 0; r < 8; r++) Sts32(col_sa + uint32_t(r * kRS * 4), uint32_t(out[r]));
        __syncwarp();
        if (m.y >> 24) {
            const uint4 lo = Lds128(row_sa), hi = Lds128(row_sa + 16);   // row j
            in[0] = int(lo.x); in[1] = int(lo.y); in[2] = int(lo.z); in[3] = int(lo.w);
            in[4] = int(hi.x); in[5] = int(hi.y); in[6] = int(hi.z); in[7] = int(hi.w);
            Islow8<18>(in, out, (1 << 17) + (128 << 18));
            const int bx = ti.bx0 + b;
            uint8_t* dst = ti.out + size_t(j) * ti.pitch + size_t(bx) * 8;
            const uint2 v = make_uint2(PackSat4(out[0], out[1], out[2], out[3]), PackSat4(out[4], out[5], out[6], out[7]));
            if (!ti.direct) {
                *reinterpret_cast<uint2*>(dst) = v;
            } else if (j < ti.clip_rows) {
                StoreClipped(dst, v, ti.clip_w - bx * 8);
            }
        }
        __syncwarp();
    }
}

}  // namespace

cudaError_t LaunchK2Idct(const K2Args& a, cudaStream_t stream) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(k2_idct, dim3((a.total_tiles + kTilesPerCta - 1) / kTilesPerCta), dim3(kThreads), 0, stream, a);
}

// Forces the module holding this stage's kernels onto the device (CUDA loads lazily: the first launch
// of every kernel would otherwise pay for it inside the first decode call).
cudaError_t PreloadK2() {
    cudaFuncAttributes at;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k2_idct);
    return e;
}

}  // namespace rjb
