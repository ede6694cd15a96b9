// idct_core.cuh — the IDCT stage's block transform, shared by k2_idct.cu, the reduced-size kernels (k2_scaled.cu)
// and the fused IDCT + output kernels (k23_fused.cu): libjpeg's jidctint.c islow butterfly (CONST_BITS 13,
// PASS1_BITS 2), bit-exact with libjpeg-turbo's jpeg_idct_islow on encoder-produced data, as BASELINE.json mandates.
// The reference delegates this to the VCN fixed-function engine (src/rocjpeg_vaapi_decoder.cpp:677-689, 816-828).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "stages.h"

namespace rjb {
namespace idct {

// shared memory through 32-bit window addresses kept in registers (the generic-pointer forms made the compiler re-derive
// the window base inside the issue-bound block loops)
__device__ __forceinline__ uint32_t SharedU32(const void* p) {
    uint32_t a = uint32_t(__cvta_generic_to_shared(p));
    asm volatile("mov.u32 %0, %0;" : "+r"(a));   // opaque: keeps the address in a register instead of re-deriving the window base
    return a;
}
__device__ __forceinline__ uint32_t Lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 Lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void Sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void Sts64(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory"); }
__device__ __forceinline__ void Sts128(uint32_t a, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// zig-zag position -> natural (row-major) position
__device__ __constant__ const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,
                                                     12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
                                                     35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51,
                                                     58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// One 8-point pass of the islow IDCT. `bias` (rounding, and in the second pass the +128
// level shift) is added to the even part once instead of to each of the 8 outputs.
template <int SHIFT>
__device__ __forceinline__ void Islow8(const int (&i)[8], int (&o)[8], int bias) {
    int z1 = (i[2] + i[6]) * 4433;
    const int t2 = z1 - i[6] * 15137;
    const int t3 = z1 + i[2] * 6270;
    const int t0 = (i[0] + i[4]) * 8192 + bias;
    const int t1 = (i[0] - i[4]) * 8192 + bias;
    const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
    int a = i[7], b = i[5], c = i[3], d = i[1];
    z1 = a + d;
    int z2 = b + c, z3 = a + c, z4 = b + d;
    const int z5 = (z3 + z4) * 9633;
    a *= 2446; b *= 16819; c *= 25172; d *= 12299;
    z1 *= -7373; z2 *= -20995;
    z3 = z3 * -16069 + z5;
    z4 = z4 * -3196 + z5;
    a += z1 + z3; b += z2 + z4; c += z2 + z3; d += z1 + z4;
    o[0] = (t10 + d) >> SHIFT; o[7] = (t10 - d) >> SHIFT;
    o[1] = (t11 + c) >> SHIFT; o[6] = (t11 - c) >> SHIFT;
    o[2] = (t12 + b) >> SHIFT; o[5] = (t12 - b) >> SHIFT;
    o[3] = (t13 + a) >> SHIFT; o[4] = (t13 - a) >> SHIFT;
}

// d = sat_u8(v0) | sat_u8(v1) << 8 | sat_u8(v2) << 16 | sat_u8(v3) << 24
__device__ __forceinline__ uint32_t PackSat4(int v0, int v1, int v2, int v3) {
    uint32_t hi, d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(hi) : "r"(v3), "r"(v2), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(v1), "r"(v0), "r"(hi));
    return d;
}

// Full-size transform of one block by 8 threads, thread j owning column j and then row j of the block's workspace
// [row][col]: row stride kRS = 12 words, block stride kBS = 104 words. A warp holds 4 blocks x 8 threads: column-wise,
// thread (b, j) touches word 104 b + 12 r + j -> bank 8 b + j + const, all 32 distinct; row-wise it moves its row as two
// 128-bit accesses whose bank groups 3 j mod 8 are distinct within each quarter-warp.
constexpr int kRS = 12, kBS = 104;

// Table entry of zig-zag code `code` (entries carry position + 1, huff_core.cuh) for the natural-order quantiser table
// qt: byte offset of the coefficient inside a block's workspace | quantiser step << 16 - one shared load replaces the
// zig-zag lookup, the row / column split and the quantiser load. Code 1 = position 0: DC-difference and pad entries,
// whose block's integrated DC goes in with the zero fill instead, are parked in a padding word of the first row.
__device__ __forceinline__ uint32_t TabEntry(int code, const uint16_t* qt) {
    const int nat = kZigzag[(code + 63) & 63];
    return uint32_t(code == 1 ? 8 * 4 : ((nat >> 3) * kRS + (nat & 7)) * 4) | (uint32_t(__ldg(qt + nat)) << 16);
}

// First half, thread j of the block whose workspace starts at blk_sa: zero fill (the dequantised integrated DC `dc` goes in
// with it), the n entries expanded into the workspace and dequantised through the table at tab_sa0 + tab_off (thread j takes ep[0],
// ep[8], ..., ep = the block's first entry + j; four loads in flight, 32 entries per block, before the first is used),
// column pass over column j. Ends with the warp synchronised for the row pass.
__device__ __forceinline__ void ScatterColumns(uint32_t blk_sa, uint32_t row_sa, uint32_t col_sa, int j, uint32_t tab_sa0, uint32_t tab_off, const uint32_t* ep, uint32_t n, uint32_t dc) {
    const uint32_t k = uint32_t(j);
    uint32_t e[4];
#pragma unroll
    for (int u = 0; u < 4; u++) e[u] = (k + 8u * u < n) ? __ldg(ep + 8 * u) : 0u;
    Sts128(row_sa, make_uint4(j == 0 ? dc : 0u, 0u, 0u, 0u));
    Sts128(row_sa + 16, make_uint4(0u, 0u, 0u, 0u));
    __syncwarp();
    const uint32_t tab_sa = tab_sa0 + tab_off;
    auto put = [&](uint32_t en) {
        const uint32_t t = Lds32(tab_sa + ((en >> 14) & 0xFCu));
        Sts32(blk_sa + (t & 0xFFFFu), uint32_t(int(int16_t(en & 0xFFFFu)) * int(t >> 16)));
    };
#pragma unroll
    for (int u = 0; u < 4; u++)
        if (k + 8u * u < n) put(e[u]);
    for (uint32_t kk = k + 32u; kk < n; kk += 8) put(__ldg(ep + (kk - k)));
    __syncwarp();
    int in[8], out[8];
#pragma unroll
    for (int r = 0; r < 8; r++) in[r] = int(Lds32(col_sa + uint32_t(r * kRS * 4)));
    Islow8<11>(in, out, 1 << 10);
#pragma unroll
    for (int r = 0; r < 8; r++) Sts32(col_sa + uint32_t(r * kRS * 4), uint32_t(out[r]));
    __syncwarp();
}

// Second half: the row pass over row j of the block (row_sa: its address in the workspace), +128 level shift included.
// The samples are packed and saturated by PackRow, which the caller places: the k23 kernels pack only valid blocks' rows.
__device__ __forceinline__ void RowPass(uint32_t row_sa, int (&out)[8]) {
    const uint4 lo = Lds128(row_sa), hi = Lds128(row_sa + 16);
    const int in[8] = {int(lo.x), int(lo.y), int(lo.z), int(lo.w), int(hi.x), int(hi.y), int(hi.z), int(hi.w)};
    Islow8<18>(in, out, (1 << 17) + (128 << 18));
}

// the row's 8 samples, saturated, packed
__device__ __forceinline__ uint2 PackRow(const int (&out)[8]) {
    return make_uint2(PackSat4(out[0], out[1], out[2], out[3]), PackSat4(out[4], out[5], out[6], out[7]));
}

}  // namespace idct
}  // namespace rjb
