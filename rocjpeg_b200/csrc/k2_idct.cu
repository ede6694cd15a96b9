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
    __shared__ __align__(16) int ws[kBlocksPerTile * kBS];
    __shared__ TileInfo s_tile[kTilesPerCta];
    __shared__ uint32_t s_tab[kTilesPerCta][64];   // per tile and zig-zag code of an entry: TabEntry
    __shared__ uint32_t s_tile0[kSearchCache];
    __shared__ __align__(16) uint4 s_meta[kTilesPerCta][kBlocksPerTile];   // per tile and block: TileBlockMeta
    static_assert((kTilesPerCta * kBlocksPerTile) % kThreads == 0, "whole record fetches per thread");
    const int tid = threadIdx.x;
    ResolveCtaTiles<8, kThreads, kTilesPerCta>(a, s_tile, s_tile0);
    for (int idx = tid; idx < kTilesPerCta * 64; idx += kThreads) {
        const int t = idx >> 6, code = idx & 63;
        const TileInfo& ti = s_tile[t];
        if (ti.nbx >= 0) s_tab[t][code] = TabEntry(code, ti.qt);
    }
    __syncthreads();
    const int b = tid >> 3, j = tid & 7;
    // Records of ALL the CTA's tiles first: every thread fetches the record pair of one (tile, block) -
    // eight tiles x 32 blocks = 256 - so the tile loop below starts from shared memory instead of
    // waiting for a dependent global load at the top of every tile (profiles/r01g_*).
#pragma unroll
    for (int rep = 0; rep < kTilesPerCta * kBlocksPerTile / kThreads; rep++) {
        const int t = (tid >> 5) + rep * (kThreads / 32), bb = tid & 31;
        s_meta[t][bb] = TileBlockMeta(s_tile[t], bb);
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
        ScatterColumns(my_sa, row_sa, col_sa, j, tab_sa0, uint32_t(it * 256), ti.entries + m.x + uint32_t(j), m.y & 0xFFFFu, m.z);
        if (m.y >> 24) {
            int out[8];
            RowPass(row_sa, out);
            const int bx = ti.bx0 + b;
            uint8_t* dst = ti.out + size_t(j) * ti.pitch + size_t(bx) * 8;
            const uint2 v = PackRow(out);
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

cudaError_t LaunchK2Idct(const K2Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(launches, k2_idct, dim3((a.total_tiles + kTilesPerCta - 1) / kTilesPerCta), dim3(kThreads), 0, stream, a);
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
