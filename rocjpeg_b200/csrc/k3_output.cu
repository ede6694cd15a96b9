// k3_output.cu — fused chroma upsampling + colour conversion + output layout (K3), sm_100a.
//
// One kernel replaces the reference's 14 post-processing kernels and its
// CopyChannel memcpys (src/rocjpeg_hip_kernels.cpp:52-2233,
// src/rocjpeg_decoder.cpp:372-636): it reads the decoded component planes at
// their coded resolution and writes the caller's buffers directly in the
// requested RocJpegOutputFormat, for every image of a batch in one launch.
//
// Arithmetic is the reference's, bit for bit:
//   * nearest-neighbour chroma replication (hip_kernels.cpp:585-617 for 4:4:0,
//     :947-954 for 4:2:2, :1389-1429 for 4:2:0);
//   * BT.709 full-range fmaf chains (hip_kernels.cpp:76-89):
//       R = fmaf(1.5748, V-128, Y); G = fmaf(-0.4681, V-128, fmaf(-0.1873, U-128, Y));
//       B = fmaf(1.8556, U-128, Y);
//   * saturating round-to-nearest-even float->u8 pack (hipPack, :25-30; the
//     rounding of v_cvt_pk_u8_f32 is this repository's documented convention);
//   * 4:0:0 replicates Y into R, G, B (hip_kernels.cpp:1915-1927, 1986-1991).
// Layout semantics (NATIVE surfaces, planar chroma sizes, pitch rules, ROI)
// follow src/rocjpeg_decoder.cpp:143-180 and :372-636; see orc_convert in
// oracle/jpeg_oracle.c for the ROI convention and the three reference defects
// that are deliberately not reproduced.
//
// Unlike the reference kernels (8 px x 2 rows per thread, no tail guard, reliant
// on allocation slack — samples/rocjpeg_samples_utils.h:387-392) every store is
// exact-bounds. Destination rows may start at any byte (pitch = 3*width is the
// samples' choice): each warp assembles one output row segment in shared memory
// at the destination's 16-byte phase and writes it with 128-bit stores in the
// aligned body, byte stores only in the unaligned head and tail.
#include <cuda_runtime.h>

#include "stages.h"

#include "k3_rows.cuh"

namespace rjb {
namespace {

using namespace k3;

__device__ __forceinline__ uint32_t UpperIndexK3(const uint32_t* a, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}


__global__ void __launch_bounds__(kThreads) k3_output(K3Args a) {
    PdlEntry();
    __shared__ __align__(16) uint8_t s_buf[kWarps][kRowBuf];
    __shared__ K3Job s_job;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        const uint32_t img = UpperIndexK3(a.img_tile0, uint32_t(a.nimages), blockIdx.x);
        const ImageDesc& im = a.images[img];
        const OutputDesc& od = a.outputs[img];
        const uint32_t t = blockIdx.x - a.img_tile0[img];
        K3Job j;
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
        s_job = j;
    }
    __syncthreads();
    const K3Job& j = s_job;
    const int W = j.W, H = j.H, x0 = j.x0, y0 = j.y0, css = j.css, fmt = j.fmt;
    const int sx = css == CSS_411 ? 2 : (css == CSS_422 || css == CSS_420) ? 1 : 0;   // chroma shift: 4:1:1 has one chroma sample per four pixels
    const int sy = (css == CSS_440 || css == CSS_420) ? 1 : 0;
    const bool gray = (css == CSS_400);
    uint8_t* buf = s_buf[warp];
    const int xt = j.xt, nx = j.nx, ty = j.ty;
    if (nx <= 0) return;

    if (fmt == FMT_RGB || fmt == FMT_RGB_PLANAR) {
        if (fmt == FMT_RGB && (j.dst[0] == nullptr || j.dpitch[0] == 0)) return;
        if (fmt == FMT_RGB_PLANAR && (!j.dst[0] || !j.dst[1] || !j.dst[2] || j.dpitch[0] == 0)) return;
        // fast rows need aligned plane loads and word-aligned destination rows (warp-uniform tests)
        const bool src_ok = ((x0 + xt) & 7) == 0;
        const uintptr_t bases = fmt == FMT_RGB ? reinterpret_cast<uintptr_t>(j.dst[0]) + size_t(xt) * 3
                                               : (reinterpret_cast<uintptr_t>(j.dst[0]) | reinterpret_cast<uintptr_t>(j.dst[1]) |
                                                  reinterpret_cast<uintptr_t>(j.dst[2])) + size_t(xt);
        for (int r = warp; r < kTileH; r += kWarps) {
            const int y = ty * kTileH + r;
            if (y >= H) break;
            const bool dst_ok = ((bases | (size_t(y) * j.dpitch[0])) & 3) == 0;
            if (src_ok && dst_ok) {
                if (sx == 2) RowRgbFast<2>(j, sy, gray, y, lane); else if (sx) RowRgbFast<1>(j, sy, gray, y, lane); else RowRgbFast<0>(j, sy, gray, y, lane);
            } else if (src_ok) {   // odd pitch / base: same conversion, the row leaves at the destination's alignment
                if (sx == 2) RowRgbStaged<2, false>(j, sy, gray, buf, y, lane); else if (sx) RowRgbStaged<1, false>(j, sy, gray, buf, y, lane);
                else RowRgbStaged<0, false>(j, sy, gray, buf, y, lane);
            } else {
                RowRgb(j, sx, sy, gray, buf, y, lane);
            }
        }
        return;
    }

    // ---- NATIVE / YUV_PLANAR / Y: plane copies and re-interleaving ----
    const bool native = (fmt == FMT_NATIVE);
    if (native && css == CSS_422) {
        // packed YUYV: byte k of the surface row is Y[k>>1] (k even), U[k>>2] (k%4==1), V[k>>2] (k%4==3);
        // the caller's row starts at surface byte 2*left (src/rocjpeg_decoder.cpp:384-388)
        if (j.dst[0] == nullptr || j.dpitch[0] == 0) return;
        for (int r = warp; r < kTileH; r += kWarps) {
            const int y = ty * kTileH + r;
            if (y >= H) break;
            const int Y = y0 + y;
            uint8_t* dst = j.dst[0] + size_t(y) * j.dpitch[0] + size_t(xt) * 2;
            const int phase = int(reinterpret_cast<uintptr_t>(dst) & 15);
            const uint8_t* yrow = j.p[0] + size_t(Y) * j.pitch[0];
            const uint8_t* urow = j.p[1] + size_t(Y) * j.pitch[1];
            const uint8_t* vrow = j.p[2] + size_t(Y) * j.pitch[2];
            const int n = nx * 2;
            for (int b = lane; b < n; b += 32) {
                const int k = 2 * (x0 + xt) + b;
                uint8_t v;
                if ((k & 1) == 0) v = __ldg(yrow + (k >> 1));
                else v = (k & 2) ? __ldg(vrow + (k >> 2)) : __ldg(urow + (k >> 2));
                buf[phase + b] = v;
            }
            __syncwarp();
            FlushRow(buf, phase, dst, n, lane);
            __syncwarp();
        }
        return;
    }
    // luma (every remaining format writes channel 0 = Y)
    if (j.dst[0] != nullptr && j.dpitch[0] != 0) {
        for (int r = warp; r < kTileH; r += kWarps) {
            const int y = ty * kTileH + r;
            if (y >= H) break;
            CopyRow(buf, j.p[0] + size_t(y0 + y) * j.pitch[0], x0 + xt, j.dst[0] + size_t(y) * j.dpitch[0] + xt, nx, lane);
        }
    }
    if (fmt == FMT_Y || gray) return;
    if (native && css == CSS_420) {
        // interleaved UV rows: surface byte k is U[k>>1] (k even) / V[k>>1] (k odd); the caller's row
        // starts at surface byte `left` of chroma row top>>1 (src/rocjpeg_decoder.cpp:380-388)
        if (j.dst[1] == nullptr || j.dpitch[1] == 0) return;
        const int rows = H >> 1;
        for (int r = warp; r < kTileH / 2; r += kWarps) {
            const int cy = ty * (kTileH / 2) + r;
            if (cy >= rows) break;
            uint8_t* dst = j.dst[1] + size_t(cy) * j.dpitch[1] + xt;
            const int phase = int(reinterpret_cast<uintptr_t>(dst) & 15);
            const uint8_t* urow = j.p[1] + size_t((y0 >> 1) + cy) * j.pitch[1];
            const uint8_t* vrow = j.p[2] + size_t((y0 >> 1) + cy) * j.pitch[2];
            for (int b = lane; b < nx; b += 32) {
                const int k = x0 + xt + b;
                buf[phase + b] = (k & 1) ? __ldg(vrow + (k >> 1)) : __ldg(urow + (k >> 1));
            }
            __syncwarp();
            FlushRow(buf, phase, dst, nx, lane);
            __syncwarp();
        }
        return;
    }
    // planar chroma at the coded resolution: (W>>sx) x (H>>sy) starting at (left>>sx, top>>sy).
    // 4:4:4 / 4:4:0 honour each channel's pitch; 4:2:2 / 4:2:0 use pitch[1] for both
    // (src/rocjpeg_decoder.cpp:589-590, 596-597, 600-601).
    const int cw = W >> sx, ch = H >> sy;
    const int rows_per_tile = kTileH >> sy, cols_per_tile = kTileW >> sx;
    const int cxt = (xt >> sx);
    const int cn = min(cols_per_tile, cw - cxt);
    if (cn <= 0) return;
    for (int task = warp; task < 2 * rows_per_tile; task += kWarps) {
        const int c = 1 + (task >= rows_per_tile ? 1 : 0);
        const int cy = ty * rows_per_tile + (task >= rows_per_tile ? task - rows_per_tile : task);
        const uint32_t pitch = (sx == 0) ? j.dpitch[c] : j.dpitch[1];
        if (cy >= ch || j.dst[c] == nullptr || pitch == 0) continue;
        CopyRow(buf, j.p[c] + size_t((y0 >> sy) + cy) * j.pitch[c], (x0 >> sx) + cxt, j.dst[c] + size_t(cy) * pitch + cxt, cn, lane);
    }
}

}  // namespace

cudaError_t LaunchK3Output(const K3Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(launches, k3_output, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
}

// Forces the module holding this stage's kernels onto the device (CUDA loads lazily: the first launch
// of every kernel would otherwise pay for it inside the first decode call).
cudaError_t PreloadK3() {
    cudaFuncAttributes at;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k3_output);
    if (e == cudaSuccess) e = PreloadK3Jfif();
    return e;
}

}  // namespace rjb
