// k3_rows.cuh — row routines of the output stage: chroma upsampling + colour conversion + store of one row segment.
//
// Shared by the stand-alone output kernel (k3_output.cu: planes read from the plane arena in global memory) and the
// fused IDCT + output kernel (k23_fused.cu: planes of one MCU row in shared memory). Arithmetic is the reference's,
// bit for bit (src/rocjpeg_hip_kernels.cpp:76-89, 585-617, 947-954, 1389-1429; see k3_output.cu).
// Template parameter SM = the plane pointers address shared memory (plain loads) instead of global memory (ld.global.nc).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "stages.h"

namespace rjb {
namespace k3 {

template <bool SM, class U>
__device__ __forceinline__ U Ld(const U* p) {
    if (SM) return *p;
    return __ldg(p);
}

constexpr int kTileW = kK3TileW;   // luma samples per tile row (8 per lane)
constexpr int kTileH = kK3TileH;   // rows per tile: each of the 8 warps walks kTileH / 8 of them
constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kChanBuf = kTileW + 32;      // one planar channel row + alignment phase
constexpr int kRowBuf = 3 * kChanBuf;      // >= 3 * kTileW + 32 (packed RGB row)

// hipPack convention: saturating round-to-nearest-even float -> u8 (one F2I on sm_100a).
__device__ __forceinline__ uint32_t PackU8(float f) {
    uint32_t r;
    asm("cvt.rni.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(f));
    return r;
}
__device__ __forceinline__ uint32_t Pack4(uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) {
    return __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
}
__device__ __forceinline__ float ByteF(uint32_t w, int i) { return float((w >> (8 * i)) & 0xFFu); }

// Write `n` bytes staged at buf[phase .. phase+n) to dst (dst & 15 == phase).
__device__ __forceinline__ void FlushRow(const uint8_t* buf, int phase, uint8_t* dst, int n, int lane) {
    int head = (16 - phase) & 15;
    if (head > n) head = n;
    if (lane < head) dst[lane] = buf[phase + lane];
    const int nvec = (n - head) >> 4;
    const uint4* s = reinterpret_cast<const uint4*>(buf + phase + head);
    uint4* d = reinterpret_cast<uint4*>(dst + head);
    for (int v = lane; v < nvec; v += 32) d[v] = s[v];
    const int done = head + (nvec << 4);
    if (done + lane < n) dst[done + lane] = buf[phase + done + lane];
}

// Load 8 consecutive samples of a plane row starting at column x (any alignment) as two
// little-endian words.
template <bool SM = false>
__device__ __forceinline__ uint2 Load8(const uint8_t* row, int x) {
    const uint8_t* p = row + x;
    if ((reinterpret_cast<uintptr_t>(p) & 7) == 0) return Ld<SM>(reinterpret_cast<const uint2*>(p));
    uint32_t b[8];
#pragma unroll
    for (int i = 0; i < 8; i++) b[i] = Ld<SM>(p + i);
    return make_uint2(Pack4(b[0], b[1], b[2], b[3]), Pack4(b[4], b[5], b[6], b[7]));
}

// Stage `n` bytes produced 8 per lane (two words) at buf[phase + 8*lane ..): word stores when
// the phase allows, byte stores otherwise and in the ragged last lane.
__device__ __forceinline__ void Stage8(uint8_t* buf, int phase, int lane, int n, uint2 v) {
    const int i0 = lane * 8;
    if (i0 >= n) return;
    uint8_t* o = buf + phase + i0;
    if ((phase & 3) == 0 && i0 + 8 <= n) {
        *reinterpret_cast<uint32_t*>(o) = v.x;
        *reinterpret_cast<uint32_t*>(o + 4) = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++)
            if (i0 + i < n) o[i] = uint8_t(((i < 4 ? v.x : v.y) >> (8 * (i & 3))) & 0xFFu);
    }
}

// Copy `n` bytes of one plane row (columns x .. x+n) into the caller's row.
__device__ __forceinline__ void CopyRow(uint8_t* buf, const uint8_t* src_row, int x, uint8_t* dst, int n, int lane) {
    // fast case (warp-uniform): aligned plane loads, word-aligned destination -> registers only
    if (((reinterpret_cast<uintptr_t>(src_row) + size_t(x)) & 7) == 0 && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
        const int m = n - lane * 8;
        if (m > 0) {
            const uint2 v = __ldg(reinterpret_cast<const uint2*>(src_row + x) + lane);
            uint8_t* d = dst + lane * 8;
            if (m >= 8) {
                if ((reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
                    *reinterpret_cast<uint2*>(d) = v;
                } else {
                    reinterpret_cast<uint32_t*>(d)[0] = v.x;
                    reinterpret_cast<uint32_t*>(d)[1] = v.y;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; i++)
                    if (i < m) d[i] = uint8_t(((i < 4 ? v.x : v.y) >> (8 * (i & 3))) & 0xFFu);
            }
        }
        return;
    }
    const int phase = int(reinterpret_cast<uintptr_t>(dst) & 15);
    // planes are MCU-padded (and the arena has slack): reading up to 7 samples past n is in bounds
    if (lane * 8 < n) Stage8(buf, phase, lane, n, Load8(src_row, x + lane * 8));
    __syncwarp();
    FlushRow(buf, phase, dst, n, lane);
    __syncwarp();
}

// Everything a CTA needs to know about its tile, resolved once by thread 0 (the kernel was
// dominated by per-thread setup when each warp did a single row: profiles/r01b_*).
struct K3Job {
    const uint8_t* p[3];
    uint32_t pitch[3];
    uint8_t* dst[4];
    uint32_t dpitch[4];
    int W, H, x0, y0, css, fmt, xt, nx, ty;
};

// One output row segment of RGB / RGB_PLANAR (nx pixels starting at column xt of row y).
template <bool SM = false>
__device__ __forceinline__ void RowRgb(const K3Job& j, int sx, int sy, bool gray, uint8_t* buf, int y, int lane) {
    const int nx = j.nx, xt = j.xt;
    const int Y = j.y0 + y;
    const int X = j.x0 + xt + lane * 8;    // first luma column of this lane
    const bool have = lane * 8 < nx;
    uint2 R = make_uint2(0, 0), G = R, B = R;   // 8 packed bytes per channel
    if (have) {
        const uint2 yy = Load8<SM>(j.p[0] + size_t(Y) * j.pitch[0], X);
        if (gray) {
            R = G = B = yy;   // hip_kernels.cpp:1915-1927
        } else {
            const uint8_t* urow = j.p[1] + size_t(Y >> sy) * j.pitch[1];
            const uint8_t* vrow = j.p[2] + size_t(Y >> sy) * j.pitch[2];
            // chroma bytes per luma pixel (nearest neighbour): `pair` = the 4 bytes of uu.x/vv.x
            // each serve two pixels (aligned 4:2:x fast path), otherwise one byte per pixel.
            uint2 uu, vv;
            const bool pair = (sx == 1) && ((X & 7) == 0);
            if (sx == 0) {
                uu = Load8<SM>(urow, X);
                vv = Load8<SM>(vrow, X);
            } else if (pair) {
                uu = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(urow + (X >> 1))), 0);
                vv = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(vrow + (X >> 1))), 0);
            } else {
                uint32_t ub[8], vb[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    ub[i] = Ld<SM>(urow + ((X + i) >> sx));
                    vb[i] = Ld<SM>(vrow + ((X + i) >> sx));
                }
                uu = make_uint2(Pack4(ub[0], ub[1], ub[2], ub[3]), Pack4(ub[4], ub[5], ub[6], ub[7]));
                vv = make_uint2(Pack4(vb[0], vb[1], vb[2], vb[3]), Pack4(vb[4], vb[5], vb[6], vb[7]));
            }
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t yw = h ? yy.y : yy.x;
                uint32_t r[4], g[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const float fy = ByteF(yw, i);
                    float fu, fv;
                    if (pair) {
                        fu = ByteF(uu.x, 2 * h + (i >> 1)) - 128.0f;
                        fv = ByteF(vv.x, 2 * h + (i >> 1)) - 128.0f;
                    } else {
                        fu = ByteF(h ? uu.y : uu.x, i) - 128.0f;
                        fv = ByteF(h ? vv.y : vv.x, i) - 128.0f;
                    }
                    r[i] = PackU8(fmaf(1.5748f, fv, fy));
                    g[i] = PackU8(fmaf(-0.4681f, fv, fmaf(-0.1873f, fu, fy)));
                    b[i] = PackU8(fmaf(1.8556f, fu, fy));
                }
                const uint32_t rw = Pack4(r[0], r[1], r[2], r[3]), gw = Pack4(g[0], g[1], g[2], g[3]),
                               bw = Pack4(b[0], b[1], b[2], b[3]);
                if (h) { R.y = rw; G.y = gw; B.y = bw; } else { R.x = rw; G.x = gw; B.x = bw; }
            }
        }
    }
    if (j.fmt == FMT_RGB) {
        uint8_t* dst = j.dst[0] + size_t(y) * j.dpitch[0] + size_t(xt) * 3;
        const int phase = int(reinterpret_cast<uintptr_t>(dst) & 15);
        if (have) {
            // interleave R,G,B bytes: 8 pixels -> 6 words
            uint32_t w[6];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t r = h ? R.y : R.x, g = h ? G.y : G.x, b = h ? B.y : B.x;
                w[3 * h + 0] = __byte_perm(__byte_perm(r, g, 0x1040), b, 0x3410);   // r0 g0 b0 r1
                w[3 * h + 1] = __byte_perm(__byte_perm(g, b, 0x2051), r, 0x3610);   // g1 b1 r2 g2
                w[3 * h + 2] = __byte_perm(__byte_perm(b, r, 0x3702), g, 0x3720);   // b2 r3 g3 b3
            }
            uint8_t* o = buf + phase + lane * 24;
            if ((phase & 3) == 0 && lane * 8 + 8 <= nx) {
#pragma unroll
                for (int k = 0; k < 6; k++) reinterpret_cast<uint32_t*>(o)[k] = w[k];
            } else {
#pragma unroll
                for (int k = 0; k < 24; k++)
                    if (lane * 8 + k / 3 < nx) o[k] = uint8_t((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
            }
        }
        __syncwarp();
        FlushRow(buf, phase, dst, nx * 3, lane);
    } else {
        // all three planes use pitch[0] (src/rocjpeg_decoder.cpp:526-544)
        uint8_t* dst[3];
        int phase[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            dst[c] = j.dst[c] + size_t(y) * j.dpitch[0] + xt;
            phase[c] = int(reinterpret_cast<uintptr_t>(dst[c]) & 15);
            Stage8(buf + c * kChanBuf, phase[c], lane, nx, c == 0 ? R : c == 1 ? G : B);
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 3; c++) FlushRow(buf + c * kChanBuf, phase[c], dst[c], nx, lane);
    }
    __syncwarp();
}

// ---- fast RGB rows ------------------------------------------------------------------------
// The general row routine above stages every row in shared memory so that any destination
// alignment gets 128-bit stores; it costs ~65 instructions per pixel (profiles/r01c_*), four times
// the arithmetic. When the tile's first plane column is a multiple of 8 (always, unless a crop
// starts at an odd multiple) and the destination row is at least 4-byte aligned, a lane can load
// its 8 samples per plane with one aligned load each, convert in registers and store words
// directly: no staging, no per-byte work.

// byte k of w as float, minus `bias`, exactly: the byte is dropped into the mantissa of 2^23
__device__ __forceinline__ float ByteToFloat(uint32_t w, uint32_t sel, float magic) {
    return __uint_as_float(__byte_perm(w, 0x4B000000u, sel)) - magic;
}

struct Rgb8 {
    uint2 r, g, b;   // 8 packed bytes per channel
};

// 8 pixels: yy = 8 luma bytes; chroma bytes per pixel given by (uw, vw) words and the byte
// selectors in csel (pixel i uses chroma byte csel[i] of the pair {lo, hi}).
template <int SX>
__device__ __forceinline__ Rgb8 Convert8(uint2 yy, uint2 uu, uint2 vv) {
    constexpr float kY = 8388608.0f, kC = 8388608.0f + 128.0f;
    float fu[8], fv[8];
    if (SX == 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            fu[i] = ByteToFloat(uu.x, 0x7650 + i, kC);
            fu[4 + i] = ByteToFloat(uu.y, 0x7650 + i, kC);
            fv[i] = ByteToFloat(vv.x, 0x7650 + i, kC);
            fv[4 + i] = ByteToFloat(vv.y, 0x7650 + i, kC);
        }
    } else if (SX == 1) {
#pragma unroll
        for (int i = 0; i < 4; i++) {   // chroma byte i serves pixels 2i and 2i+1
            fu[2 * i] = fu[2 * i + 1] = ByteToFloat(uu.x, 0x7650 + i, kC);
            fv[2 * i] = fv[2 * i + 1] = ByteToFloat(vv.x, 0x7650 + i, kC);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; i++) {   // 4:1:1: chroma byte i serves pixels 4i .. 4i+3
            fu[i] = ByteToFloat(uu.x, 0x7650 + (i >> 2), kC);
            fv[i] = ByteToFloat(vv.x, 0x7650 + (i >> 2), kC);
        }
    }
    uint32_t r[8], g[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const float fy = ByteToFloat(i < 4 ? yy.x : yy.y, 0x7650 + (i & 3), kY);
        r[i] = PackU8(fmaf(1.5748f, fv[i], fy));
        g[i] = PackU8(fmaf(-0.4681f, fv[i], fmaf(-0.1873f, fu[i], fy)));
        b[i] = PackU8(fmaf(1.8556f, fu[i], fy));
    }
    Rgb8 o;
    o.r = make_uint2(Pack4(r[0], r[1], r[2], r[3]), Pack4(r[4], r[5], r[6], r[7]));
    o.g = make_uint2(Pack4(g[0], g[1], g[2], g[3]), Pack4(g[4], g[5], g[6], g[7]));
    o.b = make_uint2(Pack4(b[0], b[1], b[2], b[3]), Pack4(b[4], b[5], b[6], b[7]));
    return o;
}

__device__ __forceinline__ void StoreBytes(uint8_t* d, uint2 v, int n) {   // first n (< 8) bytes of v
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (i < n) d[i] = uint8_t(((i < 4 ? v.x : v.y) >> (8 * (i & 3))) & 0xFFu);
}
__device__ __forceinline__ void Store8(uint8_t* d, uint2 v, bool al8) {   // d is 4-byte aligned at least
    if (al8) {
        *reinterpret_cast<uint2*>(d) = v;
    } else {
        reinterpret_cast<uint32_t*>(d)[0] = v.x;
        reinterpret_cast<uint32_t*>(d)[1] = v.y;
    }
}

// 8 converted pixels (the first n of them) of output row y from column x on; destination rows 4-byte aligned at least.
__device__ __forceinline__ void StoreRgb8(int fmt, uint8_t* dst0, uint8_t* dst1, uint8_t* dst2, uint32_t dpitch, int y, int x, int n, const Rgb8& o) {
    if (fmt == FMT_RGB) {
        uint8_t* d = dst0 + size_t(y) * dpitch + size_t(x) * 3;
        // interleave R,G,B bytes: 8 pixels -> 6 words
        uint32_t w[6];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t r = h ? o.r.y : o.r.x, g = h ? o.g.y : o.g.x, b = h ? o.b.y : o.b.x;
            w[3 * h + 0] = __byte_perm(__byte_perm(r, g, 0x1040), b, 0x3410);   // r0 g0 b0 r1
            w[3 * h + 1] = __byte_perm(__byte_perm(g, b, 0x2051), r, 0x3610);   // g1 b1 r2 g2
            w[3 * h + 2] = __byte_perm(__byte_perm(b, r, 0x3702), g, 0x3720);   // b2 r3 g3 b3
        }
        if (n >= 8) {
            if ((reinterpret_cast<uintptr_t>(d) & 7) == 0) {
#pragma unroll
                for (int k = 0; k < 3; k++) reinterpret_cast<uint2*>(d)[k] = make_uint2(w[2 * k], w[2 * k + 1]);
            } else {
#pragma unroll
                for (int k = 0; k < 6; k++) reinterpret_cast<uint32_t*>(d)[k] = w[k];
            }
        } else {
#pragma unroll
            for (int k = 0; k < 24; k++)
                if (k < 3 * n) d[k] = uint8_t((w[k >> 2] >> (8 * (k & 3))) & 0xFFu);
        }
    } else {
        // all three planes use pitch[0] (src/rocjpeg_decoder.cpp:526-544)
        const size_t off = size_t(y) * dpitch + size_t(x);
        uint8_t* d0 = dst0 + off;
        uint8_t* d1 = dst1 + off;
        uint8_t* d2 = dst2 + off;
        if (n >= 8) {
            const bool al8 = ((reinterpret_cast<uintptr_t>(d0) | reinterpret_cast<uintptr_t>(d1) | reinterpret_cast<uintptr_t>(d2)) & 7) == 0;
            Store8(d0, o.r, al8);
            Store8(d1, o.g, al8);
            Store8(d2, o.b, al8);
        } else {
            StoreBytes(d0, o.r, n);
            StoreBytes(d1, o.g, n);
            StoreBytes(d2, o.b, n);
        }
    }
}

// One output row segment (nx pixels from column xt of output row y), RGB or RGB_PLANAR.
// Preconditions (checked by the caller, warp-uniform): (x0 + xt) % 8 == 0, destination row(s) 4-byte aligned.
template <int SX, bool SM = false>
__device__ __forceinline__ void RowRgbFast(const K3Job& j, int sy, bool gray, int y, int lane) {
    const int nx = j.nx, xt = j.xt;
    const int n = nx - lane * 8;   // pixels this lane owns (may be <= 0 or < 8 at the right edge)
    if (n <= 0) return;
    const int Y = j.y0 + y;
    const int X = j.x0 + xt + lane * 8;
    const uint2 yy = Ld<SM>(reinterpret_cast<const uint2*>(j.p[0] + size_t(Y) * j.pitch[0] + X));
    Rgb8 o;
    if (gray) {
        o.r = o.g = o.b = yy;   // hip_kernels.cpp:1915-1927
    } else {
        const uint8_t* urow = j.p[1] + size_t(Y >> sy) * j.pitch[1];
        const uint8_t* vrow = j.p[2] + size_t(Y >> sy) * j.pitch[2];
        uint2 uu, vv;
        if (SX == 0) {
            uu = Ld<SM>(reinterpret_cast<const uint2*>(urow + X));
            vv = Ld<SM>(reinterpret_cast<const uint2*>(vrow + X));
        } else if (SX == 1) {
            uu = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(urow + (X >> 1))), 0u);
            vv = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(vrow + (X >> 1))), 0u);
        } else {
            uu = make_uint2(Ld<SM>(reinterpret_cast<const uint16_t*>(urow + (X >> 2))), 0u);
            vv = make_uint2(Ld<SM>(reinterpret_cast<const uint16_t*>(vrow + (X >> 2))), 0u);
        }
        o = Convert8<SX>(yy, uu, vv);
    }
    StoreRgb8(j.fmt, j.dst[0], j.dst[1], j.dst[2], j.dpitch[0], y, xt + lane * 8, n, o);
}


// ---- rows whose destination is not 4-byte aligned (odd pitches: samples/rocjpeg_samples_utils.h:334-392) ----
// Convert at the source's alignment as the fast rows do, park the 8 bytes per lane and plane in shared memory at
// word-aligned offsets, then write the row out at the DESTINATION's alignment: every lane assembles whole 16-byte
// destination vectors from five staged words with funnel shifts (the shift is the same for the whole row), byte stores
// only for the unaligned head and tail of the row.
// Copies `n` bytes staged at buf[0, n) (4-byte aligned, readable 8 bytes past n) to dst (any alignment).
__device__ __forceinline__ void FlushShifted(const uint8_t* buf, uint8_t* dst, int n, int lane) {
    const int phase = int(reinterpret_cast<uintptr_t>(dst) & 15);
    int head = (16 - phase) & 15;
    if (head > n) head = n;
    if (lane < head) dst[lane] = buf[lane];
    const int nvec = (n - head) >> 4;
    const uint32_t* w = reinterpret_cast<const uint32_t*>(buf + (head & ~3));
    const uint32_t sh = uint32_t(head & 3) * 8u;
    for (int v = lane; v < nvec; v += 32) {
        const uint32_t* q = w + 4 * v;
        const uint32_t a0 = q[0], a1 = q[1], a2 = q[2], a3 = q[3], a4 = q[4];
        uint4 o;
        o.x = __funnelshift_r(a0, a1, sh);
        o.y = __funnelshift_r(a1, a2, sh);
        o.z = __funnelshift_r(a2, a3, sh);
        o.w = __funnelshift_r(a3, a4, sh);
        reinterpret_cast<uint4*>(dst + head)[v] = o;
    }
    const int done = head + (nvec << 4);
    if (done + lane < n) dst[done + lane] = buf[done + lane];
}

__device__ __forceinline__ void StoreRgb8Staged(const K3Job& j, uint8_t* buf, int y, int lane, int n, const Rgb8& o);

// One output row segment like RowRgbFast (same preconditions on the source: (x0 + xt) % 8 == 0), any destination alignment.
// buf: per-warp staging, 16-byte aligned, at least 3 * (kTileW + 16) bytes.
template <int SX, bool SM>
__device__ __forceinline__ void RowRgbStaged(const K3Job& j, int sy, bool gray, uint8_t* buf, int y, int lane) {
    const int nx = j.nx, xt = j.xt;
    const int n = nx - lane * 8;
    const int Y = j.y0 + y;
    const int X = j.x0 + xt + lane * 8;
    Rgb8 o;
    o.r = o.g = o.b = make_uint2(0u, 0u);
    if (n > 0) {
        const uint2 yy = Ld<SM>(reinterpret_cast<const uint2*>(j.p[0] + size_t(Y) * j.pitch[0] + X));
        if (gray) {
            o.r = o.g = o.b = yy;
        } else {
            const uint8_t* urow = j.p[1] + size_t(Y >> sy) * j.pitch[1];
            const uint8_t* vrow = j.p[2] + size_t(Y >> sy) * j.pitch[2];
            uint2 uu, vv;
            if (SX == 0) {
                uu = Ld<SM>(reinterpret_cast<const uint2*>(urow + X));
                vv = Ld<SM>(reinterpret_cast<const uint2*>(vrow + X));
            } else if (SX == 1) {
                uu = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(urow + (X >> 1))), 0u);
                vv = make_uint2(Ld<SM>(reinterpret_cast<const uint32_t*>(vrow + (X >> 1))), 0u);
            } else {
                uu = make_uint2(Ld<SM>(reinterpret_cast<const uint16_t*>(urow + (X >> 2))), 0u);
                vv = make_uint2(Ld<SM>(reinterpret_cast<const uint16_t*>(vrow + (X >> 2))), 0u);
            }
            o = Convert8<SX>(yy, uu, vv);
        }
    }
    StoreRgb8Staged(j, buf, y, lane, n, o);
}

// The store half of RowRgbStaged: the lane's 8 converted pixels (the first n of them; none when n <= 0) of output row y,
// every lane of the warp calling, written out at the destination's alignment. Also the store of k3_jfif.cu's rows whose
// destination is not 4-byte aligned.
__device__ __forceinline__ void StoreRgb8Staged(const K3Job& j, uint8_t* buf, int y, int lane, int n, const Rgb8& o) {
    const int nx = j.nx, xt = j.xt;
    constexpr int kPlane = kTileW + 16;   // staged bytes per plane (+ the words FlushShifted reads past the end)
    if (j.fmt == FMT_RGB) {
        if (n > 0) {
            uint32_t w[6];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t r = h ? o.r.y : o.r.x, g = h ? o.g.y : o.g.x, b = h ? o.b.y : o.b.x;
                w[3 * h + 0] = __byte_perm(__byte_perm(r, g, 0x1040), b, 0x3410);   // r0 g0 b0 r1
                w[3 * h + 1] = __byte_perm(__byte_perm(g, b, 0x2051), r, 0x3610);   // g1 b1 r2 g2
                w[3 * h + 2] = __byte_perm(__byte_perm(b, r, 0x3702), g, 0x3720);   // b2 r3 g3 b3
            }
            uint32_t* s = reinterpret_cast<uint32_t*>(buf) + lane * 6;
#pragma unroll
            for (int k = 0; k < 6; k++) s[k] = w[k];
        }
        __syncwarp();
        FlushShifted(buf, j.dst[0] + size_t(y) * j.dpitch[0] + size_t(xt) * 3, nx * 3, lane);
    } else {
        if (n > 0) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const uint2 v = c == 0 ? o.r : c == 1 ? o.g : o.b;
                uint32_t* s = reinterpret_cast<uint32_t*>(buf + c * kPlane) + lane * 2;
                s[0] = v.x;
                s[1] = v.y;
            }
        }
        __syncwarp();
        // all three planes use pitch[0] (src/rocjpeg_decoder.cpp:526-544)
#pragma unroll
        for (int c = 0; c < 3; c++) FlushShifted(buf + c * kPlane, j.dst[c] + size_t(y) * j.dpitch[0] + xt, nx, lane);
    }
    __syncwarp();
}

}  // namespace k3
}  // namespace rjb
