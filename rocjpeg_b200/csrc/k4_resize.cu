// k4_resize.cu — Pillow's resize of decoded pictures (K4), sm_100a.
//
// Two launches per lane over all its pictures, with the arithmetic of Pillow's ImagingResampleHorizontal_8bpc /
// ImagingResampleVertical_8bpc (src/libImaging/Resample.c): per output sample and channel an int32 sum that starts
// at 1 << 21, one multiply-add per tap with the 22-bit fixed-point weights of resample.cpp, then `acc >> 22` clipped
// to 0..255. No sum can overflow: 255 * sum |w| < 2^31 for every filter. The horizontal pass runs first over the
// source rows the vertical pass reads (Pillow's ybox) and leaves 8-bit intermediate rows, exactly as Pillow does; an
// axis that keeps its size gets the one-tap identity table ((2^21 + v * 2^22) >> 22 = v), so every picture runs
// both passes.
#include <cuda_runtime.h>

#include "stages.h"

#include "k3_rows.cuh"

namespace rjb {
namespace {

constexpr int kRound = 1 << 21;

__device__ __forceinline__ uint32_t UpperIndexK4(const uint32_t* a, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ uint32_t Clip8(int acc) { return uint32_t(min(max(acc >> 22, 0), 255)); }

// One warp per intermediate row, kResizeRowsH rows per CTA, kResizeTileW output samples per tile: each lane makes the
// samples lane, lane + 32, ... of its row, every channel. The source row segment a tile reads is a few KiB that the
// warp's taps revisit, so it is read through L1 in place (staging it in shared memory behind a CTA barrier, one row per
// CTA, made every CTA a latency-bound load -> barrier -> compute chain: 0.35 ms for c3's pass on a B200); the weights of
// an output sample are the same for the CTA's eight rows.
__global__ void __launch_bounds__(kResizeThreads) k4_resize_h(K4Args a) {
    PdlEntry();
    const uint32_t ji = UpperIndexK4(a.h_tile0, uint32_t(a.njobs), blockIdx.x);
    const ResizeJob& j = a.jobs[ji];
    const int ch = j.ch, out_w = j.out_w;
    const uint32_t t = blockIdx.x - __ldg(a.h_tile0 + ji);
    const uint32_t tiles_x = uint32_t(out_w + kResizeTileW - 1) / kResizeTileW;
    const int r = int(t / tiles_x) * kResizeRowsH + (int(threadIdx.x) >> 5), xt = int(t % tiles_x) * kResizeTileW;
    if (r >= j.rows) return;
    const int nx = min(kResizeTileW, out_w - xt);
    const int2* bounds = reinterpret_cast<const int2*>(a.coef + j.h_coef);
    const int32_t* taps = a.coef + j.h_coef + 2 * out_w;
    const uint8_t* row = j.src + size_t(j.y0 + r) * j.src_pitch;
    uint8_t* orow = j.tmp + size_t(r) * j.tmp_pitch;
    for (int i = int(threadIdx.x) & 31; i < nx; i += 32) {
        const int x = xt + i;
        const int2 b = __ldg(bounds + x);
        const int32_t* k = taps + size_t(x) * size_t(j.h_ksize);
        const uint8_t* p = row + b.x * ch;
        if (ch == 3) {
            int acc0 = kRound, acc1 = kRound, acc2 = kRound;
            for (int q = 0; q < b.y; q++) {
                const int w = __ldg(k + q);
                acc0 += int(__ldg(p + 3 * q)) * w;
                acc1 += int(__ldg(p + 3 * q + 1)) * w;
                acc2 += int(__ldg(p + 3 * q + 2)) * w;
            }
            orow[3 * x] = uint8_t(Clip8(acc0));
            orow[3 * x + 1] = uint8_t(Clip8(acc1));
            orow[3 * x + 2] = uint8_t(Clip8(acc2));
        } else {
            int acc = kRound;
            for (int q = 0; q < b.y; q++) acc += int(__ldg(p + q)) * __ldg(k + q);
            orow[x] = uint8_t(Clip8(acc));
        }
    }
}

// One warp: 256 output samples of one output row, 8 per lane. Every tap is one intermediate row, read along the row
// (8 samples per lane: 24 or 8 bytes, coalesced over the warp); the weights are the same for the whole row. The
// results leave through the output stage's stores (k3_rows.cuh): registers straight to 4-byte aligned destination
// rows, staged in shared memory and written at the destination's alignment otherwise.
__global__ void __launch_bounds__(kResizeThreads) k4_resize_v(K4Args a) {
    PdlEntry();
    constexpr int kWarps = kResizeThreads / 32;
    __shared__ __align__(16) uint8_t s_buf[kWarps][k3::kRowBuf];
    const int warp = int(threadIdx.x) >> 5, lane = int(threadIdx.x) & 31;
    const uint32_t tile = blockIdx.x * kWarps + uint32_t(warp);
    if (tile >= a.v_tiles) return;
    const uint32_t ji = UpperIndexK4(a.v_tile0, uint32_t(a.njobs), tile);
    const ResizeJob& j = a.jobs[ji];
    const int ch = j.ch, out_w = j.out_w;
    const uint32_t t = tile - __ldg(a.v_tile0 + ji);
    const uint32_t tiles_x = uint32_t(out_w + kResizeTileW - 1) / kResizeTileW;
    const int y = int(t / tiles_x), xt = int(t % tiles_x) * kResizeTileW;
    const int nx = min(kResizeTileW, out_w - xt);
    const int2 b = __ldg(reinterpret_cast<const int2*>(a.coef + j.v_coef) + y);
    const int32_t* k = a.coef + j.v_coef + 2 * j.out_h + size_t(y) * size_t(j.v_ksize);
    const int n = nx - lane * 8;   // samples this lane owns (<= 0 or < 8 at the right edge)
    const int x = xt + lane * 8;
    uint8_t* buf = s_buf[warp];
    // (the intermediate rows are padded to 64 bytes and the region has slack: the loads of a ragged last lane stay inside it)
    const uint8_t* col = j.tmp + size_t(b.x - j.y0) * j.tmp_pitch + size_t(x) * ch;
    if (ch == 3) {
        int acc[24];
#pragma unroll
        for (int m = 0; m < 24; m++) acc[m] = kRound;
        if (n > 0) {
            for (int q = 0; q < b.y; q++) {
                const int w = __ldg(k + q);
                const uint2* src = reinterpret_cast<const uint2*>(col + size_t(q) * j.tmp_pitch);
#pragma unroll
                for (int v = 0; v < 3; v++) {
                    const uint2 d = __ldg(src + v);
#pragma unroll
                    for (int m = 0; m < 8; m++) acc[8 * v + m] += int(((m < 4 ? d.x : d.y) >> (8 * (m & 3))) & 0xFFu) * w;
                }
            }
        }
        // interleaved r g b bytes -> the output stage's per-channel words
        k3::Rgb8 o;
        uint32_t c8[3][8];
#pragma unroll
        for (int m = 0; m < 24; m++) c8[m % 3][m / 3] = Clip8(acc[m]);
        o.r = make_uint2(k3::Pack4(c8[0][0], c8[0][1], c8[0][2], c8[0][3]), k3::Pack4(c8[0][4], c8[0][5], c8[0][6], c8[0][7]));
        o.g = make_uint2(k3::Pack4(c8[1][0], c8[1][1], c8[1][2], c8[1][3]), k3::Pack4(c8[1][4], c8[1][5], c8[1][6], c8[1][7]));
        o.b = make_uint2(k3::Pack4(c8[2][0], c8[2][1], c8[2][2], c8[2][3]), k3::Pack4(c8[2][4], c8[2][5], c8[2][6], c8[2][7]));
        const uintptr_t bases = j.fmt == FMT_RGB ? reinterpret_cast<uintptr_t>(j.dst[0]) + size_t(xt) * 3
                                                 : (reinterpret_cast<uintptr_t>(j.dst[0]) | reinterpret_cast<uintptr_t>(j.dst[1]) |
                                                    reinterpret_cast<uintptr_t>(j.dst[2])) + size_t(xt);
        if (((bases | (size_t(y) * j.dst_pitch)) & 3) == 0) {   // warp-uniform
            if (n > 0) k3::StoreRgb8(j.fmt, j.dst[0], j.dst[1], j.dst[2], j.dst_pitch, y, x, min(n, 8), o);
        } else {
            k3::K3Job sj;
            sj.fmt = j.fmt;
            sj.xt = xt;
            sj.nx = nx;
            for (int c = 0; c < 3; c++) sj.dst[c] = j.dst[c];
            sj.dpitch[0] = j.dst_pitch;
            k3::StoreRgb8Staged(sj, buf, y, lane, n, o);
        }
        return;
    }
    int acc[8];
#pragma unroll
    for (int m = 0; m < 8; m++) acc[m] = kRound;
    if (n > 0) {
        for (int q = 0; q < b.y; q++) {
            const int w = __ldg(k + q);
            const uint2 d = __ldg(reinterpret_cast<const uint2*>(col + size_t(q) * j.tmp_pitch));
#pragma unroll
            for (int m = 0; m < 8; m++) acc[m] += int(((m < 4 ? d.x : d.y) >> (8 * (m & 3))) & 0xFFu) * w;
        }
    }
    const uint2 v = make_uint2(k3::Pack4(Clip8(acc[0]), Clip8(acc[1]), Clip8(acc[2]), Clip8(acc[3])),
                               k3::Pack4(Clip8(acc[4]), Clip8(acc[5]), Clip8(acc[6]), Clip8(acc[7])));
    uint8_t* d = j.dst[0] + size_t(y) * j.dst_pitch + xt;
    if ((reinterpret_cast<uintptr_t>(d) & 3) == 0) {   // warp-uniform
        if (n >= 8) k3::Store8(d + lane * 8, v, (reinterpret_cast<uintptr_t>(d) & 7) == 0);
        else if (n > 0) k3::StoreBytes(d + lane * 8, v, n);
    } else {
        if (n > 0) {
            reinterpret_cast<uint32_t*>(buf)[2 * lane] = v.x;
            reinterpret_cast<uint32_t*>(buf)[2 * lane + 1] = v.y;
        }
        __syncwarp();
        k3::FlushShifted(buf, d, nx, lane);
    }
}

}  // namespace

cudaError_t LaunchK4Resize(const K4Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.njobs == 0) return cudaSuccess;
    constexpr uint32_t kWarps = kResizeThreads / 32;
    cudaError_t e = LaunchPdl(launches, k4_resize_h, dim3(a.h_tiles), dim3(kResizeThreads), 0, stream, a);
    if (e == cudaSuccess) e = LaunchPdl(launches, k4_resize_v, dim3((a.v_tiles + kWarps - 1) / kWarps), dim3(kResizeThreads), 0, stream, a);
    return e;
}

cudaError_t PreloadK4() {
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, k4_resize_h);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k4_resize_v);
    return e;
}

}  // namespace rjb
