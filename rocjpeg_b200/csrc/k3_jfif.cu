// k3_jfif.cu — the output stage of RGB / RGB_PLANAR under the libjpeg colour convention (ROCJPEG_B200_COLOR_LIBJPEG), sm_100a.
//
// Produces libjpeg-turbo's default decode (what Pillow and torchvision's CPU decoder return), bit for bit, from the same
// component planes k3_output.cu reads:
//   * chroma upsampling as jdsample.c's jinit_upsampler chooses it, per picture (OutputDesc::upsample, decoder.cpp):
//       h2v1_fancy  (4:2:2)  even column 2i: (3 c[i] + c[i-1] + 1) >> 2, odd column 2i+1: (3 c[i] + c[i+1] + 2) >> 2;
//       h1v2_fancy  (4:4:0)  upper row: (3 c[k] + c[k-1] + 1) >> 2, lower row: (3 c[k] + c[k+1] + 2) >> 2;
//       h2v2_fancy  (4:2:0)  colsum = 3 c[k] + c[k-1] (upper row) or 3 c[k] + c[k+1] (lower row), then
//                            (3 colsum[i] + colsum[i-1] + 8) >> 4 (even column) and (3 colsum[i] + colsum[i+1] + 7) >> 4 (odd);
//       replication otherwise (4:4:4, 4:1:1, a 1x1 transform at scale 1/8, fancy 2x1 / 2x2 with a downsampled width <= 2);
//     a neighbour index is clamped into the picture's downsampled size (ceil(W h / hmax) x ceil(H v / vmax)), which is
//     where libjpeg duplicates edge samples: the MCU padding the IDCT writes is never read, and a crop reads the samples
//     around it (the IDCT stage transforms the blocks one chroma sample beyond the crop: k2_tile.cuh);
//   * jdcolor.c's ycc_rgb_convert: R = y + ((91881 cr + 32768) >> 16), G = y + ((-22554 cb - 46802 cr + 32768) >> 16),
//     B = y + ((116130 cb + 32768) >> 16) with cb, cr minus 128, each clamped to 0..255; 4:0:0 replicates Y.
// Same tiles (kTileW x kTileH luma samples per CTA), crop and pitch rules as k3_output; each lane makes 8 pixels of a row,
// integer arithmetic only, and stores them with k3_rows.cuh's register path (destination rows 4-byte aligned) or its
// staged path at the destination's alignment.
#include <cuda_runtime.h>

#include "stages.h"

#include "k3_rows.cuh"

namespace rjb {
namespace {

using namespace k3;

struct JfifJob {
    K3Job j;
    int cw, ch;      // the picture's downsampled chroma size
    int sx, sy;      // chroma shifts
    int mode;        // UpsampleMode
};

__device__ __forceinline__ uint32_t UpperIndexJ(const uint32_t* a, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ int Clamp255(int v) { return min(max(v, 0), 255); }

// Chroma of the lane's 8 pixels (columns X .. X+7) of one plane. row: chroma row k of the output row; nb: its vertical
// neighbour (upper row: k-1, lower row: k+1, clamped; unused without vertical fancy upsampling); lower: the output row is
// the lower one of its pair. ODD: X is odd (warp-uniform: X = x0 + xt + 8 lane).
template <int MODE, int SX, int ODD>
__device__ __forceinline__ void Chroma8(const uint8_t* row, const uint8_t* nb, int X, int cw, bool lower, int out[8]) {
    if (MODE == UP_H1V2) {
        const int bias = lower ? 2 : 1;
#pragma unroll
        for (int p = 0; p < 8; p++) {
            const int c = min(X + p, cw - 1);
            out[p] = (3 * int(__ldg(row + c)) + int(__ldg(nb + c)) + bias) >> 2;
        }
    } else if (MODE == UP_H2V1 || MODE == UP_H2V2) {
        // columns b-1 .. b+4 (b = X >> 1) hold every sample and neighbour of the 8 pixels
        const int b = X >> 1;
        int cs[6];
#pragma unroll
        for (int t = 0; t < 6; t++) {
            const int c = min(max(b - 1 + t, 0), cw - 1);
            cs[t] = MODE == UP_H2V2 ? 3 * int(__ldg(row + c)) + int(__ldg(nb + c)) : int(__ldg(row + c));
        }
        constexpr int kEven = MODE == UP_H2V2 ? 8 : 1, kOdd = MODE == UP_H2V2 ? 7 : 2, kShift = MODE == UP_H2V2 ? 4 : 2;
#pragma unroll
        for (int p = 0; p < 8; p++) {
            const int w = 1 + ((p + ODD) >> 1);   // window index of chroma column (X + p) >> 1
            out[p] = ((p + ODD) & 1) ? (3 * cs[w] + cs[w + 1] + kOdd) >> kShift : (3 * cs[w] + cs[w - 1] + kEven) >> kShift;
        }
    } else {
#pragma unroll
        for (int p = 0; p < 8; p++) out[p] = __ldg(row + min((X + p) >> SX, cw - 1));
    }
}

// The lane's 8 pixels of output row y (luma row Y = y0 + y of the picture) under the libjpeg convention.
template <int MODE, int SX, int ODD>
__device__ __forceinline__ Rgb8 Pixels8(const JfifJob& J, int y, int X) {
    const K3Job& j = J.j;
    const int Y = j.y0 + y;
    const uint2 yy = Load8(j.p[0] + size_t(Y) * j.pitch[0], X);
    Rgb8 o;
    if (j.css == CSS_400) {
        o.r = o.g = o.b = yy;
        return o;
    }
    const bool vfancy = MODE == UP_H1V2 || MODE == UP_H2V2;
    const int k = Y >> J.sy;
    const bool lower = vfancy && (Y & 1);
    const int kn = !vfancy ? k : lower ? min(k + 1, J.ch - 1) : max(k - 1, 0);
    int cb[8], cr[8];
    Chroma8<MODE, SX, ODD>(j.p[1] + size_t(k) * j.pitch[1], j.p[1] + size_t(kn) * j.pitch[1], X, J.cw, lower, cb);
    Chroma8<MODE, SX, ODD>(j.p[2] + size_t(k) * j.pitch[2], j.p[2] + size_t(kn) * j.pitch[2], X, J.cw, lower, cr);
    uint32_t r[8], g[8], b[8];
#pragma unroll
    for (int p = 0; p < 8; p++) {
        const int yv = int(((p < 4 ? yy.x : yy.y) >> (8 * (p & 3))) & 0xFFu);
        const int u = cb[p] - 128, v = cr[p] - 128;
        r[p] = uint32_t(Clamp255(yv + ((91881 * v + 32768) >> 16)));
        g[p] = uint32_t(Clamp255(yv + ((-22554 * u - 46802 * v + 32768) >> 16)));
        b[p] = uint32_t(Clamp255(yv + ((116130 * u + 32768) >> 16)));
    }
    o.r = make_uint2(Pack4(r[0], r[1], r[2], r[3]), Pack4(r[4], r[5], r[6], r[7]));
    o.g = make_uint2(Pack4(g[0], g[1], g[2], g[3]), Pack4(g[4], g[5], g[6], g[7]));
    o.b = make_uint2(Pack4(b[0], b[1], b[2], b[3]), Pack4(b[4], b[5], b[6], b[7]));
    return o;
}

// Every row of the CTA's tile that this warp owns, for one (mode, chroma shift, column parity).
template <int MODE, int SX, int ODD>
__device__ __forceinline__ void TileRows(const JfifJob& J, uint8_t* buf, int warp, int lane) {
    const K3Job& j = J.j;
    const int n = j.nx - lane * 8;   // pixels this lane owns (may be <= 0 or < 8 at the right edge)
    const int X = j.x0 + j.xt + lane * 8;
    const uintptr_t bases = j.fmt == FMT_RGB ? reinterpret_cast<uintptr_t>(j.dst[0]) + size_t(j.xt) * 3
                                             : (reinterpret_cast<uintptr_t>(j.dst[0]) | reinterpret_cast<uintptr_t>(j.dst[1]) |
                                                reinterpret_cast<uintptr_t>(j.dst[2])) + size_t(j.xt);
    for (int r = warp; r < kTileH; r += kWarps) {
        const int y = j.ty * kTileH + r;
        if (y >= j.H) break;
        Rgb8 o;
        o.r = o.g = o.b = make_uint2(0u, 0u);
        if (n > 0) o = Pixels8<MODE, SX, ODD>(J, y, X);
        if (((bases | (size_t(y) * j.dpitch[0])) & 3) == 0) {   // warp-uniform
            if (n > 0) StoreRgb8(j.fmt, j.dst[0], j.dst[1], j.dst[2], j.dpitch[0], y, j.xt + lane * 8, n, o);
        } else {
            StoreRgb8Staged(j, buf, y, lane, n, o);
        }
    }
}

template <int MODE, int SX>
__device__ __forceinline__ void TileRowsParity(const JfifJob& J, uint8_t* buf, int warp, int lane) {
    if ((J.j.x0 + J.j.xt) & 1) TileRows<MODE, SX, 1>(J, buf, warp, lane); else TileRows<MODE, SX, 0>(J, buf, warp, lane);
}

__global__ void __launch_bounds__(kThreads) k3_jfif(K3Args a) {
    PdlEntry();
    __shared__ __align__(16) uint8_t s_buf[kWarps][kRowBuf];
    __shared__ JfifJob s_job;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        const uint32_t img = UpperIndexJ(a.img_tile0, uint32_t(a.nimages), blockIdx.x);
        const ImageDesc& im = a.images[img];
        const OutputDesc& od = a.outputs[img];
        const uint32_t t = blockIdx.x - a.img_tile0[img];
        JfifJob J;
        K3Job& j = J.j;
        for (int c = 0; c < 3; c++) {
            j.p[c] = a.planes + im.plane_off[c < im.ncomp ? c : 0];
            j.pitch[c] = im.plane_pitch[c < im.ncomp ? c : 0];
        }
        for (int c = 0; c < 4; c++) {
            j.dst[c] = od.dst[c];
            j.dpitch[c] = od.dst_pitch[c];
        }
        j.W = od.w; j.H = od.h; j.x0 = od.x0; j.y0 = od.y0; j.css = im.css; j.fmt = od.fmt;
        j.xt = int(t % od.tiles_x) * kTileW;
        j.ty = int(t / od.tiles_x);
        j.nx = min(kTileW, od.w - j.xt);
        J.sx = im.css == CSS_411 ? 2 : (im.css == CSS_422 || im.css == CSS_420) ? 1 : 0;
        J.sy = (im.css == CSS_440 || im.css == CSS_420) ? 1 : 0;
        J.cw = (od.pic_w + (1 << J.sx) - 1) >> J.sx;
        J.ch = (od.pic_h + (1 << J.sy) - 1) >> J.sy;
        J.mode = od.upsample;
        s_job = J;
    }
    __syncthreads();
    const JfifJob& J = s_job;
    const K3Job& j = J.j;
    if (j.nx <= 0) return;
    if (j.fmt == FMT_RGB && (j.dst[0] == nullptr || j.dpitch[0] == 0)) return;
    if (j.fmt == FMT_RGB_PLANAR && (!j.dst[0] || !j.dst[1] || !j.dst[2] || j.dpitch[0] == 0)) return;
    uint8_t* buf = s_buf[warp];
    switch (J.mode) {
        case UP_H2V2: TileRowsParity<UP_H2V2, 1>(J, buf, warp, lane); break;
        case UP_H2V1: TileRowsParity<UP_H2V1, 1>(J, buf, warp, lane); break;
        case UP_H1V2: TileRows<UP_H1V2, 0, 0>(J, buf, warp, lane); break;
        default:
            // replication (and 4:0:0, which reads no chroma)
            if (J.sx == 2) TileRows<UP_REPLICATE, 2, 0>(J, buf, warp, lane);
            else if (J.sx == 1) TileRows<UP_REPLICATE, 1, 0>(J, buf, warp, lane);
            else TileRows<UP_REPLICATE, 0, 0>(J, buf, warp, lane);
            break;
    }
}

}  // namespace

cudaError_t LaunchK3Jfif(const K3Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(launches, k3_jfif, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
}

cudaError_t PreloadK3Jfif() {
    cudaFuncAttributes at;
    return cudaFuncGetAttributes(&at, k3_jfif);
}

}  // namespace rjb
