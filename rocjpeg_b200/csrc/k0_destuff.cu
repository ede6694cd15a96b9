// k0_destuff.cu — GPU pass over the raw entropy-coded bytes (K0), sm_100a.
//
// Takes over, for a whole batch per launch, the per-byte work of the reference's parser - the
// byte-serial search for FF D9 (RocJpegStreamParser::ParseEOI, src/rocjpeg_parser.cpp:400-416) -
// and what the VCN engine does with the slice it is handed (src/rocjpeg_vaapi_decoder.cpp:681:
// the hardware strips byte stuffing and restart markers itself). The host parser stops at the
// end of the SOS header; the bytes behind it are uploaded untouched and this pass
//   * finds the end of the slice (first FF D9),
//   * removes byte stuffing (FF 00 -> FF), fill bytes (FF FF) and restart markers (FF D0..D7),
//   * discovers the restart intervals and writes the batch's segment table (SegmentDesc),
//   * writes the destuffed bytes of interval k at SegmentStart(r_k, k, S) of the image's clean
//     stream (device_types.h) followed by 16 zero bytes - the layout K1 decodes from.
// Rules for damaged streams are those of the host restatement (jpeg_parser.cpp:
// ExtractEntropyData), which is also the expected value in the tests: any other marker inside an
// interval ends that interval's data; intervals beyond the frame's count are dropped; a lone FF
// at the end carries no data.
//
// Formulation. Whether byte p is kept, ends an interval, ends the slice or kills the interval
// depends on bytes p-1, p, p+1 only. Where it goes depends on a prefix over everything before it:
//   (restart markers so far, kept bytes since the last one, position behind the last one,
//    interval dead, slice ended)
// which composes associatively (Combine below), so three launches do it: per-tile reduction,
// one scan over the tiles of each image, per-tile scan + scatter. A tile is 16 KiB of one image,
// four 16-byte pieces (64 consecutive bytes) per thread. When the upload is the gather kernel
// (many small pictures read in place from page-locked host memory), the per-tile reduction rides
// in it: the bytes pass through the SMs anyway while the PCIe link is the limit. The kernels are
// issue-bound, not bandwidth-bound (the batch's raw bytes sit in L2), hence: a thread whose 64
// bytes hold no FF - four out of five - is recognised with two instructions per word and does no
// classification at all; a warp without markers scans one integer instead of the four-word
// element; kept bytes leave through shared memory as 128-bit stores, one run per restart interval.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "k0_core.cuh"
#include "stages.h"

namespace rjb {
namespace {

using namespace k0;

constexpr int kThreads = 256;
constexpr int kPieces = 4;                      // 16-byte pieces per thread
constexpr int kChunk = 16 * kPieces;            // bytes per thread
constexpr int kTileBytes = kK0TileBytes;
static_assert(kTileBytes == kThreads * kChunk, "64 bytes per thread");
constexpr int kStageBytes = 32 * kChunk + 48;   // a warp's kept bytes at the run's 16-byte phase

__device__ __forceinline__ Elem ShflUp(const Elem& e, int d) {
    Elem r;
    r.nrst = __shfl_up_sync(0xFFFFFFFFu, e.nrst, d);
    r.tail = __shfl_up_sync(0xFFFFFFFFu, e.tail, d);
    r.last_r = __shfl_up_sync(0xFFFFFFFFu, e.last_r, d);
    r.flags = __shfl_up_sync(0xFFFFFFFFu, e.flags, d);
    return r;
}

__device__ __forceinline__ Elem ShflDown(const Elem& e, int d) {
    Elem r;
    r.nrst = __shfl_down_sync(0xFFFFFFFFu, e.nrst, d);
    r.tail = __shfl_down_sync(0xFFFFFFFFu, e.tail, d);
    r.last_r = __shfl_down_sync(0xFFFFFFFFu, e.last_r, d);
    r.flags = __shfl_down_sync(0xFFFFFFFFu, e.flags, d);
    return r;
}

// A thread's 64 bytes of an image's uploaded data.
//   kind kGeneral  anything else: a marker of any kind (FF not followed by 00), two stuffed bytes in one word, or a chunk
//                  that reaches over an end of the scan - the per-piece code of k0_core.cuh handles it;
//   kind kData     wholly inside the scan, no FF in it, the byte before it is not FF: 64 data bytes;
//   kind kStuffed  wholly inside the scan, every FF in it is followed by 00 (byte stuffing only): the data bytes are the
//                  chunk minus the bytes that follow an FF. `drop[i]` flags those (0x80 in the byte's lane), at most one per word.
// Four chunks out of five are kData, nearly all others kStuffed; both are recognised and counted without a branch per byte.
enum ChunkKind : int { kGeneral = 0, kData = 1, kStuffed = 2 };
struct Chunk {
    uint32_t w[4 * kPieces];
    uint32_t drop[4 * kPieces];
    uint32_t prev, next;   // the bytes around it (only meaningful inside the scan)
    int64_t pos0;          // scan position of byte 0
    bool overlaps;         // some byte lies inside the scan
    int kind;
    uint32_t nkeep;        // data bytes of a kData / kStuffed chunk
};

// 0x80 in every byte of x that is zero (exact per byte: no carries between bytes)
__device__ __forceinline__ uint32_t ZeroBytes(uint32_t x) { return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u; }

__device__ __forceinline__ void FinishChunk(Chunk& c, int64_t len) {
    constexpr int NW = 4 * kPieces;
    c.overlaps = c.pos0 + kChunk > 0 && c.pos0 < len;
    c.kind = kGeneral;
    c.nkeep = 0;
    if (!(c.pos0 >= 0 && c.pos0 + kChunk <= len)) return;
    uint32_t f[NW], any = 0, ev = 0, two = 0, holes = 0;
#pragma unroll
    for (int i = 0; i < NW; i++) {
        f[i] = ZeroBytes(~c.w[i]);   // FF bytes
        any |= f[i];
    }
    if (any == 0u && c.prev != 0xFFu) {
        c.kind = kData;
        c.nkeep = kChunk;
        return;
    }
#pragma unroll
    for (int i = 0; i < NW; i++) {
        // the byte that follows each byte of word i, lane for lane
        const uint32_t nb = i + 1 < NW ? __funnelshift_r(c.w[i], c.w[i + 1], 8) : ((c.w[i] >> 8) | (c.next << 24));
        ev |= f[i] & ~ZeroBytes(nb);                                                             // FF followed by something else than 00
        const uint32_t d = (i ? __funnelshift_l(f[i - 1], f[i], 8) : ((f[0] << 8) | (c.prev == 0xFFu ? 0x80u : 0u))) & ~f[i];   // bytes behind an FF (an FF there is judged on its own)
        c.drop[i] = d;
        two |= d & (d - 1u);
        holes += uint32_t(__popc(d));
    }
    // (the byte behind an FF in front of the chunk is dropped whatever it is - stuffing or the second byte of a marker
    // that belongs to the previous chunk - unless it is FF itself, which `ev` then reports)
    if ((ev | two) == 0u) {
        c.kind = kStuffed;
        c.nkeep = uint32_t(kChunk) - holes;
    }
}

// `off` = byte offset of the chunk in the image's uploaded bytes (multiple of 64).
__device__ __forceinline__ Chunk LoadChunk(const uint8_t* raw, const ImageDesc& im, uint64_t off) {
    Chunk c;
    const int64_t len = int64_t(im.raw_len);
    c.pos0 = int64_t(off) - int64_t(im.raw_skip);
    c.prev = 0u;
    c.next = 0xFFu;
    const uint8_t* base = raw + im.raw_off + off;
#pragma unroll
    for (int j = 0; j < kPieces; j++) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (PieceOverlaps(c.pos0 + 16 * j, len)) v = __ldg(reinterpret_cast<const uint4*>(base) + j);
        c.w[4 * j] = v.x; c.w[4 * j + 1] = v.y; c.w[4 * j + 2] = v.z; c.w[4 * j + 3] = v.w;
    }
    if (c.pos0 > 0 && c.pos0 <= len) c.prev = __ldg(base - 1);
    if (c.pos0 + kChunk < len && c.pos0 + kChunk >= 0) c.next = __ldg(base + kChunk);
    FinishChunk(c, len);
    return c;
}

__device__ __forceinline__ Piece PieceOf(const Chunk& c, int j, int64_t len) {
    const uint32_t prev = j ? (c.w[4 * j - 1] >> 24) : c.prev;
    const uint32_t next = j < kPieces - 1 ? (c.w[4 * j + 4] & 0xFFu) : c.next;
    return ClassifyPiece(*reinterpret_cast<const uint32_t(*)[4]>(&c.w[4 * j]), prev, next, c.pos0 + 16 * j, len);
}

// The chunk's prefix element; *plain = it holds no marker (the element is just a byte count).
__device__ __forceinline__ Elem ChunkElem(const Chunk& c, int64_t len, bool* plain) {
    Elem e{0u, 0u, 0u, 0u};
    *plain = true;
    if (c.kind != kGeneral) {
        e.tail = c.nkeep;
        return e;
    }
    if (!c.overlaps) return e;
#pragma unroll
    for (int j = 0; j < kPieces; j++) {
        const Piece pc = PieceOf(c, j, len);
        if (!pc.any) continue;
        e = Combine(e, PieceElem(pc));
        if (pc.rst | pc.oth | pc.eoi) *plain = false;
    }
    return e;
}

// largest i in [0, n) with a[i] <= v
__device__ __forceinline__ uint32_t UpperIndexK0(const uint32_t* a, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// Scan of `e` over the CTA: *excl = exclusive value of the thread, *total = CTA total (when asked for).
// `plain` = the thread's chunk holds no marker: a warp (a CTA) of plain chunks - nearly all of them when the
// picture has no restart markers - scans one integer instead of four words through Combine.
__device__ __forceinline__ void CtaScan(const Elem& e, bool plain, Elem* warp_tot /* shared [kThreads / 32] */, Elem* excl, Elem* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Elem inc = e;
    const bool warp_plain = __all_sync(0xFFFFFFFFu, plain);
    if (warp_plain) {
        uint32_t t = e.tail;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t p = __shfl_up_sync(0xFFFFFFFFu, t, d);
            if (lane >= d) t += p;
        }
        inc.tail = t;
    } else {
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const Elem p = ShflUp(inc, d);
            if (lane >= d) inc = Combine(p, inc);
        }
    }
    if (lane == 31) warp_tot[warp] = inc;
    Elem ex = ShflUp(inc, 1);
    if (lane == 0) ex = Elem{0u, 0u, 0u, 0u};
    if (__syncthreads_and(warp_plain)) {
        uint32_t pre = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; w++) {
            const uint32_t t = warp_tot[w].tail;
            if (w < warp) pre += t;
            tot += t;
        }
        ex.tail += pre;
        *excl = ex;
        if (total) *total = Elem{0u, tot, 0u, 0u};
        return;
    }
    Elem pre{0u, 0u, 0u, 0u};
    for (int w = 0; w < warp; w++) pre = Combine(pre, warp_tot[w]);
    *excl = Combine(pre, ex);
    if (total) {
        Elem t = pre;
        for (int w = warp; w < kThreads / 32; w++) t = Combine(t, warp_tot[w]);
        *total = t;
    }
}

// ---------------------------------------------------------------- k0_reduce: one element per tile

__global__ void __launch_bounds__(kThreads) k0_reduce(K0Args a) {
    PdlEntry();
    __shared__ Elem s_warp[kThreads / 32];
    const uint32_t tile = blockIdx.x;
    const uint32_t img = UpperIndexK0(a.img_tile0, uint32_t(a.nimages), tile);
    const ImageDesc& im = a.images[img];
    const uint64_t off = uint64_t(tile - im.k0_tile0) * kTileBytes + uint64_t(threadIdx.x) * kChunk;
    const Chunk c = LoadChunk(a.raw, im, off);
    bool plain;
    const Elem e = ChunkElem(c, int64_t(im.raw_len), &plain);
    Elem ex, tot;
    CtaScan(e, plain, s_warp, &ex, &tot);
    if (threadIdx.x == 0) {
        a.tile_sum[tile] = make_uint4(tot.nrst, tot.tail, tot.last_r, tot.flags);
        if (tile == im.k0_tile0) a.status[img] = ScanStatus{0u, 0u, 0u, 0u};   // the later passes OR their findings into it
    }
}

// ---------------------------------------------------------------- gather_reduce: upload + k0_reduce in one
//
// Many small pictures in page-locked host memory: a few CTAs copy them, 16 KiB at a time, straight from the
// caller's buffers into the raw arena (a copy call per picture would cost the host more than the transfer).
// The link is the limit, so the tile's prefix element is computed on the way, from the copy kept in shared
// memory - the separate reduction launch (and its read of the bytes) is not needed then.

constexpr int kGatherCtas = 64;   // PCIe-bound: a few CTAs saturate the link; the rest of the GPU stays free
                                  // for the kernels of the other pipeline lanes

__global__ void __launch_bounds__(kThreads) gather_reduce(K0Args a, const GatherItem* items, uint8_t* raw_out) {
    PdlEntry();
    __shared__ Elem s_warp[kThreads / 32];
    __shared__ __align__(16) uint4 s_tile[kTileBytes / 16];
    __shared__ uint32_t s_edge[2];
    const int tid = threadIdx.x;
    for (uint32_t tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
        const uint32_t img = UpperIndexK0(a.img_tile0, uint32_t(a.nimages), tile);
        const ImageDesc& im = a.images[img];
        const GatherItem it = items[img];
        const uint32_t off = (tile - im.k0_tile0) * uint32_t(kTileBytes);
        const uint32_t n = it.nbytes > off ? min(uint32_t(kTileBytes), it.nbytes - off) : 0u;   // multiple of 16
        const int64_t len = int64_t(im.raw_len), tpos0 = int64_t(off) - int64_t(im.raw_skip);
        __syncthreads();   // the previous tile's readers of s_tile / s_edge / s_warp are done
        // the bytes around the tile, read from the source (the neighbouring tiles are other CTAs' work)
        if (tid == 0) s_edge[0] = (tpos0 > 0 && tpos0 <= len) ? uint32_t(it.src[off - 1]) : 0u;
        if (tid == 32) s_edge[1] = (tpos0 + kTileBytes < len) ? uint32_t(it.src[off + kTileBytes]) : 0xFFu;
        const uint4* src = reinterpret_cast<const uint4*>(it.src + off);
        uint4* dst = reinterpret_cast<uint4*>(raw_out + it.dst_off + off);
        for (uint32_t i = uint32_t(tid); i < uint32_t(kTileBytes / 16); i += kThreads) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (i < n / 16) {
                v = src[i];
                dst[i] = v;
            }
            s_tile[i] = v;
        }
        __syncthreads();
        Chunk c;
        c.pos0 = tpos0 + int64_t(tid) * kChunk;
#pragma unroll
        for (int j = 0; j < kPieces; j++) {
            const uint4 v = s_tile[tid * kPieces + j];
            c.w[4 * j] = v.x; c.w[4 * j + 1] = v.y; c.w[4 * j + 2] = v.z; c.w[4 * j + 3] = v.w;
        }
        c.prev = tid ? (reinterpret_cast<const uint32_t*>(s_tile)[tid * (kChunk / 4) - 1] >> 24) : s_edge[0];
        c.next = tid < kThreads - 1 ? (reinterpret_cast<const uint32_t*>(s_tile)[(tid + 1) * (kChunk / 4)] & 0xFFu) : s_edge[1];
        if (c.pos0 <= 0) c.prev = 0u;
        if (c.pos0 + kChunk >= len) c.next = 0xFFu;
        FinishChunk(c, len);
        bool plain;
        const Elem e = ChunkElem(c, len, &plain);
        Elem ex, tot;
        CtaScan(e, plain, s_warp, &ex, &tot);
        if (tid == 0) {
            a.tile_sum[tile] = make_uint4(tot.nrst, tot.tail, tot.last_r, tot.flags);
            if (tile == im.k0_tile0) a.status[img] = ScanStatus{0u, 0u, 0u, 0u};
        }
    }
}

// ---------------------------------------------------------------- k0_scan: exclusive scan over an image's tiles

__global__ void __launch_bounds__(kThreads) k0_scan(K0Args a) {
    PdlEntry();
    __shared__ Elem s_warp[kThreads / 32];
    const uint32_t img = blockIdx.x;
    const uint32_t t0 = a.img_tile0[img], t1 = a.img_tile0[img + 1];
    Elem carry{0u, 0u, 0u, 0u};
    for (uint32_t base = t0; base < t1; base += kThreads) {
        const uint32_t k = base + threadIdx.x;
        Elem e{0u, 0u, 0u, 0u};
        if (k < t1) {
            const uint4 q = a.tile_sum[k];
            e = Elem{q.x, q.y, q.z, q.w};
        }
        Elem ex, tot;
        __syncthreads();   // the previous chunk's readers of s_warp are done
        CtaScan(e, false, s_warp, &ex, &tot);
        ex = Combine(carry, ex);
        if (k < t1) a.tile_carry[k] = make_uint4(ex.nrst, ex.tail, ex.last_r, ex.flags);
        carry = Combine(carry, tot);
    }
}

// ---------------------------------------------------------------- k0_apply: scatter + segment table

struct DevMem {
    const K0Args& a;
    const ImageDesc& im;
    uint32_t img;
    uint32_t* fill_from;   // shared: first restart interval the bytes do not contain
    __device__ __forceinline__ SegmentDesc& Segment(uint32_t k) const { return a.segments[im.seg0 + k]; }
    __device__ __forceinline__ uint8_t* Clean() const { return a.clean + im.data_off; }
    __device__ __forceinline__ void Flag(uint32_t bits) const {
        if (bits) atomicOr(&a.status[img].flags, bits);
    }
    __device__ __forceinline__ void Finish(uint32_t segments_seen, uint32_t scan_size, uint32_t from) const {
        a.status[img].segments_seen = segments_seen;
        a.status[img].scan_size = scan_size;
        *fill_from = from;
    }
};

// Removes the dropped bytes of a kStuffed chunk in registers: from the top word down (a deletion only moves what lies
// above it, which has been dealt with), the bytes above a hole slide down by one. Afterwards the first c.nkeep bytes of
// w[] are the chunk's data bytes in order.
__device__ __forceinline__ void DeleteHoles(Chunk& c) {
    constexpr int NW = 4 * kPieces;
#pragma unroll
    for (int i = NW - 1; i >= 0; i--) {
        const uint32_t d = c.drop[i];
        if (d) {
            const uint32_t below = (d >> 7) - 1u;                                   // the bytes of word i below the hole (d = 0x80 << 8b)
            const uint32_t up = i + 1 < NW ? c.w[i + 1] : 0u;
            c.w[i] = (c.w[i] & below) | (__funnelshift_r(c.w[i], up, 8) & ~below);   // hole closed, the next word's first byte enters
#pragma unroll
            for (int k = i + 1; k < NW; k++) c.w[k] = __funnelshift_r(c.w[k], k + 1 < NW ? c.w[k + 1] : 0u, 8);
        }
    }
}

// The first n bytes of the NW little-endian words w[] to shared memory at byte address `at` (any alignment), exactly:
// whole words of the stream as seen from the destination's word grid (funnel-shifted), byte stores only for the words
// the run covers partly at its two ends - a neighbouring lane owns their other bytes.
template <int NW>
__device__ __forceinline__ void StoreBytesShifted(uint8_t* at, const uint32_t (&w)[NW], uint32_t n) {
    const uint32_t a = uint32_t(reinterpret_cast<uintptr_t>(at)) & 3u;
    uint32_t* p = reinterpret_cast<uint32_t*>(at - a);
    const uint32_t sh = 32u - 8u * a;   // (funnel shifts take their count mod 32: a == 0 passes w[k] through)
#pragma unroll
    for (int k = 0; k <= NW; k++) {
        // destination word k holds stream bytes [4k - a, 4k - a + 4)
        const uint32_t lo_w = k ? w[k - 1] : 0u, hi_w = k < NW ? w[k] : 0u;
        const uint32_t v = a ? __funnelshift_r(lo_w, hi_w, sh) : hi_w;
        const int lo = 4 * k - int(a), hi = lo + 4;
        if (lo >= 0 && hi <= int(n)) {
            if (k < NW || a) p[k] = v;
        } else if (hi > 0 && lo < int(n)) {
#pragma unroll
            for (int b = 0; b < 4; b++)
                if (lo + b >= 0 && lo + b < int(n)) reinterpret_cast<uint8_t*>(p + k)[b] = uint8_t(v >> (8 * b));
        }
    }
}

template <int S>
__global__ void __launch_bounds__(kThreads) k0_apply(K0Args a) {
    PdlEntry();
    __shared__ Elem s_warp[kThreads / 32];
    __shared__ Elem s_carry;
    __shared__ __align__(16) uint8_t s_stage[kThreads / 32][kStageBytes];
    __shared__ uint32_t s_fill_from;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;
    const uint32_t img = UpperIndexK0(a.img_tile0, uint32_t(a.nimages), tile);
    const ImageDesc& im = a.images[img];
    const int64_t len = int64_t(im.raw_len);
    const uint64_t off = uint64_t(tile - im.k0_tile0) * kTileBytes + uint64_t(tid) * kChunk;
    Chunk c = LoadChunk(a.raw, im, off);
    bool plain;
    const Elem mine = ChunkElem(c, len, &plain);
    if (c.kind == kStuffed) DeleteHoles(c);
    Elem ex;
    if (tid == 0) s_fill_from = 0xFFFFFFFFu;
    if (a.inline_scan) {
        // no picture has more than 32 tiles: the tile combines the prefix elements of the picture's earlier tiles itself (one lane
        // each, in order) - k0_scan is not launched
        if (warp == 0) {
            const uint32_t k = im.k0_tile0 + uint32_t(lane);
            Elem e{0u, 0u, 0u, 0u};
            if (k < tile) {
                const uint4 q = a.tile_sum[k];
                e = Elem{q.x, q.y, q.z, q.w};
            }
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {   // lane i ends up with e_i o e_{i+1} o ... (the empty element is neutral)
                const Elem p = ShflDown(e, d);
                if (lane + d < 32) e = Combine(e, p);
            }
            if (lane == 0) s_carry = e;
        }
    }
    CtaScan(mine, plain, s_warp, &ex, nullptr);   // (ends with a CTA barrier: s_carry is visible behind it)
    if (a.inline_scan) {
        ex = Combine(s_carry, ex);
    } else {
        const uint4 q = a.tile_carry[tile];
        ex = Combine(Elem{q.x, q.y, q.z, q.w}, ex);
    }
    DevMem mem{a, im, img, &s_fill_from};
    const Placer<DevMem> pl{im, uint32_t(S), mem};
    const bool ended_before = (ex.flags & kEnded) != 0;

    // Chunks without a marker: their kept bytes form one contiguous piece of their restart interval, at the offset
    // the prefix gives (kept bytes since the interval began). The lanes of a warp that belong to the same
    // interval - all of them, unless a restart marker lies in the warp's 2 KiB - gather their bytes in shared
    // memory at the run's 16-byte phase and write them out as 128-bit stores.
    const uint32_t n = mine.tail;
    const bool staged = plain && c.overlaps && !ended_before && !(ex.flags & kDead) && n != 0u && pl.Wanted(ex.nrst);
    uint32_t todo = __ballot_sync(0xFFFFFFFFu, staged);
    while (todo) {
        const int leader = __ffs(int(todo)) - 1;
        const uint32_t kL = __shfl_sync(0xFFFFFFFFu, ex.nrst, leader), rL = __shfl_sync(0xFFFFFFFFu, ex.last_r, leader),
                       cL = __shfl_sync(0xFFFFFFFFu, ex.tail, leader);
        const bool member = staged && ex.nrst == kL;
        const uint32_t members = __ballot_sync(0xFFFFFFFFu, member);
        // bytes of the run (every warp-wide exchange of an iteration happens here, before the lanes go separate ways)
        const uint32_t total = __shfl_sync(0xFFFFFFFFu, ex.tail + n, 31 - __clz(int(members))) - cL;
        uint8_t* dst = pl.Dst(rL, kL) + cL;
        const uint32_t phase = uint32_t(reinterpret_cast<uintptr_t>(dst) & 15u);
        if (member) {
            uint8_t* at = s_stage[warp] + phase + (ex.tail - cL);
            if (c.kind != kGeneral) {
                StoreBytesShifted<4 * kPieces>(at, c.w, n);   // (the holes of a kStuffed chunk were deleted above)
            } else {
                // a chunk at an end of the scan, or with two stuffed bytes in one word: piece by piece, byte stores
#pragma unroll
                for (int j = 0; j < kPieces; j++) at += CompactPiece(PieceOf(c, j, len), at);
            }
        }
        __syncwarp();
        const uint8_t* buf = s_stage[warp] + phase;
        uint32_t head = (16u - phase) & 15u;
        if (head > total) head = total;
        if (uint32_t(lane) < head) dst[lane] = buf[lane];
        const uint32_t nvec = (total - head) >> 4;
        for (uint32_t v = uint32_t(lane); v < nvec; v += 32)
            reinterpret_cast<uint4*>(dst + head)[v] = reinterpret_cast<const uint4*>(buf + head)[v];
        const uint32_t done = head + (nvec << 4);
        if (done + uint32_t(lane) < total) dst[done + lane] = buf[done + lane];
        __syncwarp();
        todo &= ~members;
    }
    // Chunks with a marker walk their pieces (bytes stored one by one, restart intervals opened and closed); the first
    // chunk of the image opens interval 0; the chunk holding the last byte closes the last interval when there is no FF D9.
    // (The walk indexes the chunk's words by a run-time piece number: it reads them from the warp's staging buffer, free
    // by now, so that the register copy is only ever indexed statically and stays in registers.)
    const bool first = tile == im.k0_tile0 && tid == 0;
    const bool walk = !plain && c.overlaps && !ended_before;
    if (first) pl.Open(0u, 0u);
    if (len == 0) {
        if (first) pl.End(0u, 0u, 0u, 0u, kScanNoEoi);
    } else if (walk) {
        uint32_t* sw = reinterpret_cast<uint32_t*>(s_stage[warp]) + lane * (kChunk / 4);
#pragma unroll
        for (int k = 0; k < 4 * kPieces; k++) sw[k] = c.w[k];
        Elem x = ex;
#pragma unroll 1
        for (int j = 0; j < kPieces; j++) {
            const uint32_t prev = j ? (sw[4 * j - 1] >> 24) : c.prev;
            const uint32_t next = j < kPieces - 1 ? (sw[4 * j + 4] & 0xFFu) : c.next;
            const uint32_t pw[4] = {sw[4 * j], sw[4 * j + 1], sw[4 * j + 2], sw[4 * j + 3]};
            const Piece pc = ClassifyPiece(pw, prev, next, c.pos0 + 16 * j, len);
            const Elem pe = PieceElem(pc);
            if (pc.any && !(x.flags & kEnded)) WalkPiece(pc, x, pe, pl);
            FinishPiece(pc, x, pe, pl, false);
            x = Combine(x, pe);
        }
    } else if (plain && c.overlaps && !ended_before && c.pos0 + kChunk >= len) {
        const Elem inc = Combine(ex, mine);   // no marker in the chunk that holds the last byte: the slice ends with the buffer
        pl.End(inc.last_r, inc.nrst, inc.tail, im.raw_len, kScanNoEoi | ((inc.flags & kStray) ? kScanStrayMarker : 0u));
    }
    __syncthreads();
    const uint32_t from = s_fill_from;
    if (from != 0xFFFFFFFFu)
        for (uint32_t q = from + uint32_t(tid); q < im.nseg; q += kThreads) pl.Missing(q);
}

}  // namespace

cudaError_t LaunchK0Reduce(const K0Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(launches, k0_reduce, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
}

cudaError_t LaunchGatherReduce(const K0Args& a, const GatherItem* items, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    return LaunchPdl(launches, gather_reduce, dim3(min(a.total_tiles, uint32_t(kGatherCtas))), dim3(kThreads), 0, stream, a, items, const_cast<uint8_t*>(a.raw));
}

cudaError_t LaunchK0Destuff(const K0Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_tiles == 0) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (!a.inline_scan) e = LaunchPdl(launches, k0_scan, dim3(a.nimages), dim3(kThreads), 0, stream, a);
    if (e != cudaSuccess) return e;
    if (getenv("ROCJPEG_B200_DEBUG_SYNC")) {
        e = cudaStreamSynchronize(stream);
        fprintf(stderr, "[rocjpeg_b200] k0_reduce + k0_scan: %s\n", cudaGetErrorName(e));
        if (e != cudaSuccess) return e;
    }
    switch (a.sub_bytes) {
        case 32: return LaunchPdl(launches, k0_apply<32>, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
        case 64: return LaunchPdl(launches, k0_apply<64>, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
        case 128: return LaunchPdl(launches, k0_apply<128>, dim3(a.total_tiles), dim3(kThreads), 0, stream, a);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t PreloadK0() {
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, k0_reduce);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, gather_reduce);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k0_scan);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k0_apply<32>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k0_apply<64>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k0_apply<128>);
    return e;
}

}  // namespace rjb
