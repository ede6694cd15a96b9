// k2_scaled.cu — dequantise + reduced-size inverse DCT for decodes at scale 1/2, 1/4 and 1/8, sm_100a.
//
// The arithmetic is libjpeg's jidctred.c (the reduced IDCTs libjpeg-turbo selects with scale_num = 1,
// scale_denom = d): an 8x8 block of coefficients becomes an S x S block of samples, S = 8 / d.
//   k2_idct_4x4  jpeg_idct_4x4: CONST_BITS 13, PASS1_BITS 2; row and column 4 of the block are not used
//   k2_idct_2x2  jpeg_idct_2x2: only positions 0, 1, 3, 5, 7 of each row and column are used
//   k2_idct_1x1  jpeg_idct_1x1: (DC * q0 + 4) >> 3, +128 - reads the block record's integrated DC only
// libjpeg's shortcuts for all-zero AC columns and rows are arithmetically identical to the general path,
// so none are taken. Outputs saturate like the full-size path (PackSat4), and the intermediate
// arithmetic is 32-bit like k2_idct.cu's.
//
// Input, tiling and every rule about which blocks are transformed are those of k2_idct (k2_tile.cuh): a
// tile is 32 horizontally adjacent blocks of one block row of a component, a block's coefficient entries
// run from its predecessor's record to its own, a record that fails the validity tests contributes its
// integrated DC only. Mapping for S = 4 and 2: 4 threads per block, which share its entries and columns, the
// first S of them one output row each; a 256-thread CTA works on 2 tiles at a time. (2 threads per block at S = 2
// left each thread a serial chain of entry loads twice as long.) The entries are scattered into a
// zeroed shared-memory workspace that holds only the rows and columns the transform reads (7 x 7 at
// S = 4, 5 x 5 at S = 2); entries at positions the transform ignores go to a dump word. Mapping for
// S = 1: one thread per block, no workspace.
#include <cuda_runtime.h>

#include "idct_core.cuh"
#include "k2_tile.cuh"
#include "stages.h"

namespace rjb {
namespace {

using namespace idct;
using namespace k2tile;

constexpr int kThreads = 256;
constexpr int kTilesPerCta = 16;
constexpr int kTpb = 4;   // threads per block in the 4x4 and 2x2 kernels

// jidctred.c constants (FIX(x) = round(x * 2^13))
constexpr int kF0_211164243 = 1730, kF0_509795579 = 4176, kF0_601344887 = 4926, kF0_720959822 = 5906,
              kF0_765366865 = 6270, kF0_850430095 = 6967, kF0_899976223 = 7373, kF1_061594337 = 8697,
              kF1_272758580 = 10426, kF1_451774981 = 11893, kF1_847759065 = 15137, kF2_172734803 = 17799,
              kF2_562915447 = 20995, kF3_624509785 = 29692;

// Rows / columns of the 8x8 block the S-point transform reads, in workspace order: K of them.
template <int S> struct Kept;
template <> struct Kept<4> {
    static constexpr int K = 7;
    __device__ static int Slot(int nat) { return nat == 4 ? -1 : nat < 4 ? nat : nat - 1; }   // 0 1 2 3 5 6 7
};
template <> struct Kept<2> {
    static constexpr int K = 5;
    __device__ static int Slot(int nat) { return nat == 0 ? 0 : (nat & 1) ? (nat + 1) >> 1 : -1; }   // 0 1 3 5 7
};

// One pass of jpeg_idct_4x4 over the 7 values of a row or column (slots 0..6 = positions 0 1 2 3 5 6 7).
// `bias` carries the rounding (and in the second pass the +128 level shift).
template <int SHIFT>
__device__ __forceinline__ void Idct4(const int (&v)[7], int (&o)[4], int bias) {
    const int t0 = v[0] * (1 << 14) + bias;   // << (CONST_BITS + 1)
    const int t2 = v[2] * kF1_847759065 - v[5] * kF0_765366865;
    const int t10 = t0 + t2, t12 = t0 - t2;
    const int z1 = v[6], z2 = v[4], z3 = v[3], z4 = v[1];   // positions 7, 5, 3, 1
    const int a = -z1 * kF0_211164243 + z2 * kF1_451774981 - z3 * kF2_172734803 + z4 * kF1_061594337;
    const int b = -z1 * kF0_509795579 - z2 * kF0_601344887 + z3 * kF0_899976223 + z4 * kF2_562915447;
    o[0] = (t10 + b) >> SHIFT;
    o[3] = (t10 - b) >> SHIFT;
    o[1] = (t12 + a) >> SHIFT;
    o[2] = (t12 - a) >> SHIFT;
}

// One pass of jpeg_idct_2x2 over the 5 values of a row or column (slots 0..4 = positions 0 1 3 5 7).
template <int SHIFT>
__device__ __forceinline__ void Idct2(const int (&v)[5], int (&o)[2], int bias) {
    const int t10 = v[0] * (1 << 15) + bias;   // << (CONST_BITS + 2)
    const int t0 = -v[4] * kF0_720959822 + v[3] * kF0_850430095 - v[2] * kF1_272758580 + v[1] * kF3_624509785;
    o[0] = (t10 + t0) >> SHIFT;
    o[1] = (t10 - t0) >> SHIFT;
}

// S samples of one block row into the caller's buffer: n = visible samples left in the row
template <int S>
__device__ __forceinline__ void StoreRow(uint8_t* dst, uint32_t v, int n) {
    const uintptr_t al = reinterpret_cast<uintptr_t>(dst);
    if (n >= S && (al & (S - 1)) == 0) {
        if (S == 4) *reinterpret_cast<uint32_t*>(dst) = v;
        else if (S == 2) *reinterpret_cast<uint16_t*>(dst) = uint16_t(v);
        else *dst = uint8_t(v);
    } else {
#pragma unroll
        for (int i = 0; i < S; i++)
            if (i < n) dst[i] = uint8_t((v >> (8 * i)) & 0xFFu);
    }
}

template <int S>
__device__ __forceinline__ void ScaledBody(const K2Args& a) {
    constexpr int K = Kept<S>::K;
    constexpr int kWords = (K * K + 1 + 3) & ~3;   // workspace of a block: K x K values + a dump word, whole 16-byte vectors
    constexpr int kTilesAtOnce = kThreads / (kBlocksPerTile * kTpb);
    __shared__ __align__(16) int ws[kTilesAtOnce * kBlocksPerTile * kWords];
    __shared__ TileInfo s_tile[kTilesPerCta];
    // per tile and zig-zag code of an entry: byte offset of the coefficient inside a block's workspace (low half; the
    // dump word for positions the transform ignores) and its quantiser step (high half)
    __shared__ uint32_t s_tab[kTilesPerCta][64];
    __shared__ uint32_t s_tile0[kSearchCache];
    __shared__ __align__(16) uint4 s_meta[kTilesPerCta][kBlocksPerTile];   // per tile and block: TileBlockMeta
    const int tid = threadIdx.x;
    ResolveCtaTiles<S, kThreads, kTilesPerCta>(a, s_tile, s_tile0);
    for (int idx = tid; idx < kTilesPerCta * 64; idx += kThreads) {
        const int t = idx >> 6, code = idx & 63;   // entries carry position + 1 (huff_core.cuh)
        const TileInfo& ti = s_tile[t];
        if (ti.nbx >= 0) {
            const int nat = kZigzag[(code + 63) & 63];
            const int r = Kept<S>::Slot(nat >> 3), c = Kept<S>::Slot(nat & 7);
            // (code 1 = position 0: DC-difference and pad entries - the integrated DC comes from the record)
            const int word = (code == 1 || r < 0 || c < 0) ? K * K : r * K + c;
            s_tab[t][code] = uint32_t(word * 4) | (uint32_t(__ldg(ti.qt + nat)) << 16);
        }
    }
    // block records of all the CTA's tiles
    for (int idx = tid; idx < kTilesPerCta * kBlocksPerTile; idx += kThreads) {
        const int t = idx >> 5, bb = idx & 31;
        s_meta[t][bb] = TileBlockMeta(s_tile[t], bb);
    }
    __syncthreads();
    const int group = tid / (kBlocksPerTile * kTpb), gt = tid % (kBlocksPerTile * kTpb);
    const int b = gt / kTpb, j = gt % kTpb;   // block of the tile, thread of the block (output row j < S)
    const uint32_t blk_sa = SharedU32(ws) + uint32_t(((group * kBlocksPerTile) + b) * kWords * 4);
#pragma unroll 1
    for (int it = group; it < kTilesPerCta; it += kTilesAtOnce) {
        const TileInfo& ti = s_tile[it];
        if (ti.nbx < 0) break;
        if (ti.direct == 2) continue;
        const uint4 m = s_meta[it][b];
        const uint32_t n = m.y & 0xFFFFu;
        const uint32_t* ep = ti.entries + m.x;
        uint32_t e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) e[u] = (uint32_t(j + kTpb * u) < n) ? __ldg(ep + j + kTpb * u) : 0u;
        for (int w = j; w < kWords / 4; w += kTpb)   // zero fill; the integrated DC goes in with it
            Sts128(blk_sa + uint32_t(w * 16), make_uint4(w == 0 ? m.z : 0u, 0u, 0u, 0u));
        __syncwarp();
        const uint32_t tab_sa = SharedU32(&s_tab[it][0]);
        auto put = [&](uint32_t en) {
            const uint32_t t = Lds32(tab_sa + ((en >> 14) & 0xFCu));
            Sts32(blk_sa + (t & 0xFFFFu), uint32_t(int(int16_t(en & 0xFFFFu)) * int(t >> 16)));
        };
#pragma unroll
        for (int u = 0; u < 4; u++)
            if (uint32_t(j + kTpb * u) < n) put(e[u]);
        for (uint32_t k0 = uint32_t(j + 4 * kTpb); k0 < n; k0 += 4 * kTpb) {   // the rest four loads at a time
#pragma unroll
            for (int u = 0; u < 4; u++) e[u] = (k0 + uint32_t(kTpb * u) < n) ? __ldg(ep + k0 + kTpb * u) : 0u;
#pragma unroll
            for (int u = 0; u < 4; u++)
                if (k0 + uint32_t(kTpb * u) < n) put(e[u]);
        }
        __syncwarp();
        // pass 1: columns, descaled by CONST_BITS - PASS1_BITS + log2(8 / S); outputs overwrite the column's first S slots
#pragma unroll
        for (int c = j; c < K; c += kTpb) {
            if (S == 4) {
                int v[7], o[4];
#pragma unroll
                for (int r = 0; r < 7; r++) v[r] = int(Lds32(blk_sa + uint32_t((r * K + c) * 4)));
                Idct4<12>(v, o, 1 << 11);
#pragma unroll
                for (int r = 0; r < 4; r++) Sts32(blk_sa + uint32_t((r * K + c) * 4), uint32_t(o[r]));
            } else {
                int v[5], o[2];
#pragma unroll
                for (int r = 0; r < 5; r++) v[r] = int(Lds32(blk_sa + uint32_t((r * K + c) * 4)));
                Idct2<13>(v, o, 1 << 12);
#pragma unroll
                for (int r = 0; r < 2; r++) Sts32(blk_sa + uint32_t((r * K + c) * 4), uint32_t(o[r]));
            }
        }
        __syncwarp();
        if ((m.y >> 24) && j < S) {   // pass 2: row j, descaled by CONST_BITS + PASS1_BITS + 3 + log2(8 / S), +128, saturated
            uint32_t packed;
            if (S == 4) {
                int v[7], o[4];
#pragma unroll
                for (int c = 0; c < 7; c++) v[c] = int(Lds32(blk_sa + uint32_t((j * K + c) * 4)));
                Idct4<19>(v, o, (1 << 18) + (128 << 19));
                packed = PackSat4(o[0], o[1], o[2], o[3]);
            } else {
                int v[5], o[2];
#pragma unroll
                for (int c = 0; c < 5; c++) v[c] = int(Lds32(blk_sa + uint32_t((j * K + c) * 4)));
                Idct2<20>(v, o, (1 << 19) + (128 << 20));
                packed = PackSat4(o[0], o[1], 0, 0);
            }
            const int bx = ti.bx0 + b;
            uint8_t* dst = ti.out + size_t(j) * ti.pitch + size_t(bx) * S;
            if (!ti.direct) {
                if (S == 4) *reinterpret_cast<uint32_t*>(dst) = packed;
                else *reinterpret_cast<uint16_t*>(dst) = uint16_t(packed);
            } else if (j < ti.clip_rows) {
                StoreRow<S>(dst, packed, ti.clip_w - bx * S);
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kThreads) k2_idct_4x4(K2Args a) {
    PdlEntry();
    ScaledBody<4>(a);
}

__global__ void __launch_bounds__(kThreads) k2_idct_2x2(K2Args a) {
    PdlEntry();
    ScaledBody<2>(a);
}

// 1/8: one thread per block, the block's 8-byte record is all it reads.
__global__ void __launch_bounds__(kThreads) k2_idct_1x1(K2Args a) {
    PdlEntry();
    __shared__ TileInfo s_tile[kTilesPerCta];
    __shared__ uint32_t s_tile0[kSearchCache];
    const int tid = threadIdx.x;
    ResolveCtaTiles<1, kThreads, kTilesPerCta>(a, s_tile, s_tile0);
    const int bb = tid & 31;
#pragma unroll 1
    for (int it = tid >> 5; it < kTilesPerCta; it += kThreads / 32) {
        const TileInfo& ti = s_tile[it];
        if (ti.nbx < 0) break;
        const int bx = ti.bx0 + bb;
        if (ti.direct == 2 || bx >= ti.nbx) continue;
        const int dc = int(__ldg(&ti.rec[TileBlock(ti, bx)].dc)) * int(__ldg(ti.qt));
        const uint32_t v = PackSat4((dc + 4 + (128 << 3)) >> 3, 0, 0, 0);
        if (!ti.direct || bx < ti.clip_w) ti.out[bx] = uint8_t(v);
    }
}

}  // namespace

cudaError_t LaunchK2Scaled(const K2Args& a, int scale_denom, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    const dim3 grid((a.total_tiles + kTilesPerCta - 1) / kTilesPerCta);
    switch (scale_denom) {
        case 2: return LaunchPdl(launches, k2_idct_4x4, grid, dim3(kThreads), 0, stream, a);
        case 4: return LaunchPdl(launches, k2_idct_2x2, grid, dim3(kThreads), 0, stream, a);
        case 8: return LaunchPdl(launches, k2_idct_1x1, grid, dim3(kThreads), 0, stream, a);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t PreloadK2Scaled() {
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, k2_idct_4x4);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k2_idct_2x2);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k2_idct_1x1);
    return e;
}

}  // namespace rjb
