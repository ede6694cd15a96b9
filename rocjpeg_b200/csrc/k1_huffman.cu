// k1_huffman.cu — entropy-decode stage (K1) for sm_100a.
//
// Replaces the Huffman decoding the reference delegates to AMD's VCN
// fixed-function JPEG engine (vaRenderPicture/vaEndPicture at
// src/rocjpeg_vaapi_decoder.cpp:677-689 and :816-828). One launch covers every
// image of a batch.
//
// Work decomposition
//   segment      = one restart interval (or the whole scan when DRI is absent):
//                  byte-aligned start, known decoder state, known first block.
//   subsequence  = S consecutive bytes of a segment (S = 32/64/128), one thread.
//   CTA          = kK1Threads threads on ONE image: kK1Threads - halo consecutive subsequences
//                  it owns + the halo (2 or 4) before them (re-decoded, never stored); the
//                  image's Huffman tables and the CTA's bytes are staged in shared memory.
//
// Schedule (self-synchronising parallel Huffman decoding)
//   k1_sync round 0   (also fills the batch's block records with "never decoded")
//                     every thread decodes its subsequence from a guessed state
//                     (exact for the first subsequence of a segment) and records
//                     its end state; then, inside the CTA, every thread whose
//                     predecessor's end state differs from the state it started
//                     from re-decodes, until nothing changes. Huffman streams
//                     re-synchronise within tens of bytes, so this is typically
//                     two decodes per thread, and thanks to the halo the state
//                     entering the CTA's first owned subsequence is almost always
//                     final already.
//   k1_sync round r>0 verifies every CTA boundary against the owner's result and
//                     repairs the few that differ. A CTA whose incoming state is
//                     unchanged exits at once. The host checks the counter of the
//                     last round; a non-zero value triggers more rounds
//                     (correctness never depends on the stream synchronising).
//   k1_scan           per image: exclusive prefix of the CTAs' block counts
//                     (segmented at restart intervals) and entry counts.
//   k1_write          the final decode: the image's sparse coefficient stream (one
//                     32-bit (int16 value, zig-zag index) entry per symbol with
//                     magnitude bits, eight per 256-bit store) and one 8-byte record
//                     per block {where its entries end, DC difference}.
//   k1_fused          counting and write pass in one kernel; for pictures of up to kK1DcMaxMcus MCUs, each CTA then also
//                     integrates the DC of its share of the picture's blocks (IntegrateDc) and no DC kernel runs.
//   dc_sums / dc_scan / dc_apply
//                     per-component, per-restart-interval prefix sum of the DC
//                     differences in tiles of 256 MCUs over all SMs; the integrated DC
//                     replaces the difference in the block's record, where K2 reads it.
#include <cuda_runtime.h>

#include <cstddef>

#include "huff_core.cuh"
#include "stages.h"

namespace rjb {

namespace {

constexpr int T = kK1Threads;
constexpr uint32_t kNoState = 0xFFFFFFFFu;

// largest i in [0, n) with a[i] <= v (a is non-decreasing, a[0] <= v)
__device__ __forceinline__ uint32_t UpperIndex(const uint32_t* a, uint32_t n, uint32_t v) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// The CTA -> image search of the two decode kernels: on a copy of the prefix array in shared memory (the
// scan-word area, not yet in use) when it fits - one coalesced load instead of eight dependent ones.
template <int CAP>
__device__ __forceinline__ uint32_t ImageOfCta(const K1Args& a, uint32_t* scratch, uint32_t cta) {
    const uint32_t n = uint32_t(a.nimages);
    if (n > uint32_t(CAP)) return UpperIndex(a.img_cta0, n, cta);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) scratch[i] = __ldg(a.img_cta0 + i);
    __syncthreads();
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (scratch[mid] <= cta) lo = mid; else hi = mid;
    }
    __syncthreads();   // the area is about to be overwritten with the scan words
    return lo;
}

// ---- raw shared-memory primitives for the two hot loops ----------------------------------
__device__ __forceinline__ uint32_t SharedAddr(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint32_t Lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t Lds16(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}

// Decoder state of one thread packed so that adding a table entry (huff_core.cuh: MakeEntry)
// advances all of it at once:
//   bits 0..10   bit position inside the subsequence, biased by 1024 - (end of the subsequence
//                rounded up to a whole 32-bit word): bit 10 comes on when the position passes
//                that end (link entries use the same bit of a table entry as their mark).
//   bits 11..20  coefficient entries produced so far
//   bits 21..26  zig-zag index; bit 27 comes on with the symbol that ends a block
//   bits 28..31  scratch (the SSSS fields of the entries pile up here and fall off the top)
// Rounding the end up only matters for the last subsequence of a restart interval: the symbols
// it may see past the true end lie in the interval's zero padding, change nothing downstream
// (no hand-over; the write pass stops at the interval's last block and zero-fills what the
// counting pass reserved for them).
constexpr uint32_t kAccStop = 1u << 10;
constexpr uint32_t kAccBlockEnd = 1u << 27;
constexpr uint32_t kAccKeep = 0x001FFFFFu;   // cleared at a block end: zig-zag index, end flag, scratch
constexpr uint32_t kAccZMask = 63u << 21;

// Addresses (shared window) of everything the decode loops touch besides the thread's own slot.
struct LutView {
    uint32_t fast_sa;            // first pair's DC table; pair k at + k * 4096, its AC table 2048 further
    uint32_t sub_sa;             // second-level arena
    const HuffLutSet* set;       // global copy (canonical search for link entries with x = 0)
    const uint8_t* pair_tab;     // shared: [2 * pair + is_ac] -> table index in the set
};

// A code longer than kFastBits: second-level lookup by the x bits that follow the first kFastBits.
__device__ __forceinline__ uint32_t CanonicalSearch(const LutView& lv, uint32_t off, uint32_t win) {
    return SlowEntry(lv.set, lv.pair_tab[(off - lv.fast_sa) >> 11], win >> 16);   // off = fast_sa + 4096 * pair + 2048 * is_ac
}
__device__ __forceinline__ uint32_t ResolveLink(const LutView& lv, uint32_t e, uint32_t off, uint32_t win) {
    const uint32_t x = LinkBits(e);
    if (x == 0) return CanonicalSearch(lv, off, win);
    return Lds32(lv.sub_sa + ((LinkFirst(e) + ((win << kFastBits) >> (32u - x))) << 2));
}

// One thread's decoder registers. The three per-symbol updates are written as predicated PTX so
// that each costs a fixed, minimal number of issue slots: with 32 lanes per warp some lane
// crosses a word boundary or ends a block in almost every step, so these paths are executed by
// the warp every time whether written as branches or not (profiles/r01c_*).
//   window    w0:w1 hold the 64 bits around the read position, w2 is fetched one word ahead, so
//             the only shared-memory access on the symbol-to-symbol dependency chain is the
//             table lookup;
//   schedule  a pointer walking through the CTA's shared array of DC-table addresses, one entry
//             per block from the start of an MCU on, repeated (the block-in-MCU counter is the
//             pointer itself). A pair's AC table lies 2048 bytes after its DC table and DC tables
//             start at addresses with bit 11 clear (checked in StageCta), so "the AC table of
//             whatever table is current" is off | 2048.
struct Lane {
    uint32_t acc;              // packed state, see above
    uint32_t w0, w1, w2, wp;   // wp = shared address of w2
    uint32_t sp0, sp;          // shared address of the schedule entry of the first / current block
    uint32_t next_dc;          // DC-table address of the next block, fetched one block ahead
    uint32_t off;              // table the next symbol is looked up in

    __device__ __forceinline__ void Init(uint32_t slot_sa, uint32_t sched_sa, uint32_t key, uint32_t end_bit) {
        const uint32_t p = StateOverflow(key), end32 = (end_bit + 31u) & ~31u;
        acc = (p + 1024u - end32) | (uint32_t(StateZ(key)) << 21);
        wp = slot_sa + ((p >> 5) << 2);
        w0 = Lds32(wp);
        w1 = Lds32(wp + 4);
        w2 = Lds32(wp + 8);
        wp += 8;
        sp0 = sp = sched_sa + 2u * uint32_t(StateC(key));
        off = Lds16(sp) | (StateZ(key) ? 2048u : 0u);
        next_dc = Lds16(sp + 2);
    }
    __device__ __forceinline__ uint32_t Peek() const { return __funnelshift_l(w1, w0, acc); }
    __device__ __forceinline__ uint32_t Lookup(uint32_t win) const {
        uint32_t a, e;
        asm volatile("{\n\t.reg .b32 i;\n\tshr.u32 i, %2, 23;\n\tmad.lo.u32 %0, i, 4, %3;\n\tld.shared.u32 %1, [%0];\n\t}"
                     : "=r"(a), "=r"(e) : "r"(win), "r"(off));
        return e;
    }
    // acc <- nxt; window refill when the position entered the next word; block-end bookkeeping.
#define RJB_K1_COMMIT_HEAD(NXT)                              \
    "lop3.b32 t, %0, %" NXT ", 32, 0x28;\n\t"               \
    "setp.ne.u32 pc, t, 0;\n\t"                             \
    "and.b32 t, %" NXT ", 0x8000000;\n\t"                   \
    "setp.ne.u32 pe, t, 0;\n\t"                             \
    "@pc mov.b32 %1, %2;\n\t"                               \
    "@pc mov.b32 %2, %3;\n\t"                               \
    "@pc add.u32 %4, %4, 4;\n\t"                            \
    "@pc ld.shared.u32 %3, [%4];\n\t"                       \
    "mov.b32 %0, %" NXT ";\n\t"                             \
    "or.b32 %7, %7, 2048;\n\t"                              \
    "@pe and.b32 %0, %" NXT ", 0x1fffff;\n\t"               \
    "@pe mov.b32 %7, %6;\n\t"                               \
    "@pe add.u32 %5, %5, 2;\n\t"                            \
    "@pe ld.shared.u16 %6, [%5+2];\n\t"
    __device__ __forceinline__ void Commit(uint32_t nxt) {
        asm volatile("{\n\t.reg .pred pc, pe;\n\t.reg .b32 t;\n\t" RJB_K1_COMMIT_HEAD("8") "}"
                     : "+r"(acc), "+r"(w0), "+r"(w1), "+r"(w2), "+r"(wp), "+r"(sp), "+r"(next_dc), "+r"(off)
                     : "r"(nxt));
    }
    // The same, and at a block end: the block's record gets `n` (entries so far = one past the
    // block's last) and, when this thread decoded the block's DC symbol (always, except for a first
    // block that began in the previous subsequence), the DC difference in the same 8-byte store - one
    // scattered store per block instead of two, the store path is the write pass's second bottleneck
    // (profiles/r01d_*). The record pointer moves on; reaching the record of the restart interval's
    // last block + 1 raises the stop bit (what follows in the subsequence is padding).
    __device__ __forceinline__ void CommitWrite(uint32_t nxt, BlockRec*& rp, uint32_t n, uint32_t rp_stop, int dcv, uint32_t& has_dc) {
        asm volatile("{\n\t.reg .pred pc, pe, pl, pf, pn;\n\t.reg .b32 t;\n\t" RJB_K1_COMMIT_HEAD("10")
                     "setp.ne.and.u32 pf, %9, 0, pe;\n\t"
                     "setp.eq.and.u32 pn, %9, 0, pe;\n\t"
                     "@pf st.global.v2.b32 [%8], {%11, %13};\n\t"
                     "@pn st.global.u32 [%8], %11;\n\t"
                     "@pe mov.b32 %9, 1;\n\t"
                     "@pe add.u64 %8, %8, 8;\n\t"
                     "cvt.u32.u64 t, %8;\n\t"
                     "setp.eq.and.u32 pl, t, %12, pe;\n\t"
                     "@pl or.b32 %0, %0, 0x400;\n\t"
                     "}"
                     : "+r"(acc), "+r"(w0), "+r"(w1), "+r"(w2), "+r"(wp), "+r"(sp), "+r"(next_dc), "+r"(off), "+l"(rp), "+r"(has_dc)
                     : "r"(nxt), "r"(n), "r"(rp_stop), "r"(dcv)
                     : "memory");
    }
#undef RJB_K1_COMMIT_HEAD
    __device__ __forceinline__ uint32_t Blocks() const { return (sp - sp0) >> 1; }
};

// Count-only decode of one subsequence from state `key` (speculation / synchronisation):
// returns the packed end state + block count, the number of coefficient entries in *nnz_out.
__device__ __forceinline__ uint32_t DecodeCount(uint32_t slot_sa, const LutView& lv, uint32_t sched_sa, int bpm, uint32_t key,
                                                uint32_t end_bit, uint32_t* nnz_out) {
    Lane ln;
    ln.Init(slot_sa, sched_sa, key, end_bit);
    if (end_bit != 0) {
        for (;;) {
            const uint32_t win = ln.Peek();
            uint32_t e = ln.Lookup(win);
            if (IsLink(e)) e = ResolveLink(lv, e, ln.off, win);
            ln.Commit(ln.acc + e);
            if (ln.acc & kAccStop) break;
        }
    }
    const uint32_t nb = ln.Blocks(), acc = ln.acc;
    *nnz_out = (((acc >> 11) & 0x3FFu) + 7u) & ~7u;   // a thread's run of the entry stream is padded to whole 32-byte stores
    // bits consumed past the end: the loop stops at the end rounded up to a whole word, the successor starts at the end
    // itself (they differ for the inline-destuffed subsequences of k1_fused, whose ends fall on any byte; for the others
    // only in a restart interval's last subsequence, which hands over nothing)
    return PackState(((acc & 63u) + ((0u - end_bit) & 31u)) & 63u, int((uint32_t(StateC(key)) + nb) % uint32_t(bpm)), int((acc >> 21) & 63u), nb > 0xFFFFu ? 0xFFFFu : nb);
}

// Per-thread description of its subsequence. Subsequence g of an image covers bytes [g S, (g+1) S) of the
// image's clean stream; the destuffing pass starts every restart interval on a multiple of S
// (device_types.h: SegmentStart), so a subsequence belongs to one interval, and the few that fall into the
// gap between two intervals map to no data.
struct Sub {
    bool in_range;     // inside the image's subsequence range
    bool active;       // maps to real data
    bool first;        // first subsequence of its segment (state known exactly)
    bool last;         // last subsequence of its segment
    uint32_t seg;      // global segment index
    uint32_t end_bit;  // bits of entropy-coded data inside the subsequence
    uint64_t start;    // byte offset of the subsequence in the scan arena
};

// Segment k of the batch. Inline destuffing (no K0 ran, the table is not written): the picture's one restart interval,
// measured in raw bytes up to the FF D9 that ends the caller's buffer; subsequence g of the picture then covers raw bytes
// [g S, (g+1) S) of its entropy-coded data, and StageInline turns them into at most S destuffed bytes. (INL: compiled for
// inline destuffing - the instance of k1_fused that LaunchK1Fused picks when K1Args::inline_destuff is set; every other
// kernel, and k1_fused for the lanes that keep K0, has none of it.)
template <bool INL>
__device__ __forceinline__ SegmentDesc SegmentOf(const K1Args& a, const ImageDesc& im, uint32_t k) {
    if (!INL) return a.segments[k];
    SegmentDesc sd;
    sd.data_off = im.data_off;
    sd.nbytes = im.raw_len - 2u;
    sd.sub0 = im.sub0;
    sd.blk_first = 0;
    sd.blk_count = im.nblocks;
    return sd;
}

template <int S, bool INL>
__device__ __forceinline__ Sub Locate(const K1Args& a, const ImageDesc& im, int64_t gi, bool use_cache) {
    Sub s;
    s.in_range = s.active = gi >= int64_t(im.sub0) && gi < int64_t(im.sub0) + int64_t(im.nsub);
    s.first = s.last = false;
    s.seg = 0;
    s.end_bit = 0;
    s.start = 0;
    if (!s.active) return s;
    const uint32_t g = uint32_t(gi);
    uint32_t k;
    if (use_cache) {
        k = a.sub_seg[g];
    } else {
        // segments of this image: [seg0, seg0 + nseg), ordered by sub0
        uint32_t lo = 0, hi = im.nseg;
        while (hi - lo > 1) {
            uint32_t mid = (lo + hi) >> 1;
            if (__ldg(&a.segments[im.seg0 + mid].sub0) <= g) lo = mid; else hi = mid;
        }
        k = im.seg0 + lo;
    }
    const SegmentDesc sd = SegmentOf<INL>(a, im, k);
    const uint32_t j = g - sd.sub0;
    const uint32_t nchunks = (sd.nbytes + S - 1) / S;
    s.seg = k;
    s.active = j < nchunks;   // behind the interval's last byte (or the interval is empty / not wanted): no data
    s.first = (j == 0);
    s.last = (j + 1 >= nchunks);
    const uint32_t off = j * S;
    const uint32_t remain = sd.nbytes > off ? sd.nbytes - off : 0;
    s.end_bit = (remain < uint32_t(S) ? remain : uint32_t(S)) * 8u;
    s.start = sd.data_off + off;
    return s;
}

// Shared-memory image of one CTA's working set. Dynamic shared memory starts with the Huffman
// tables (4 KiB per table pair the image uses + the second-level arena: K1Args::lut_smem_bytes,
// the batch maximum), this struct follows. Every byte counts: at 32 KiB per CTA seven CTAs fit an
// SM instead of six, and the two decode kernels are latency-bound (profiles/r01c_c3_kernels.md).
template <int S>
struct K1Smem {
    static constexpr int kSlotVecs = (S + 16) / 16;      // 16-byte vectors staged per subsequence
    static constexpr int kSlotStride = S / 4 + 3;        // words kept: subsequence + 12 bytes of look-ahead (a symbol is at
                                                         // most 31 bits, the window prefetches two words); the stride is odd:
                                                         // conflict-free when lanes read the same word index
    static constexpr int kSchedLen = S * 4 + 48;         // a block takes at least 2 bits: S*4 blocks + one MCU + prefetch
    uint32_t words[T * kSlotStride + 1];                 // + the word the last slot's final vector spills
    uint32_t start[T];                                   // byte offset of the subsequence from the image's data_off (~0: none)
    uint32_t state[T];
    uint32_t used[T];
    uint32_t nnz[T];
    uint32_t endbit[T];
    uint32_t queue[T];
    uint16_t sched[kSchedLen];
    uint8_t pair_tab[8];
    uint32_t scratch[40];
};

// Huffman tables + block schedule of one image into shared memory (any CTA size; no barrier inside).
template <int S>
__device__ __forceinline__ LutView StageTables(uint32_t* lut, uint16_t* sched, uint8_t* pair_tab, const K1Args& a, const ImageDesc& im) {
    const int tid = threadIdx.x, nth = blockDim.x;
    // Lane forms "AC table of the current pair" as (table address | 2048): every pair's DC table must
    // start at a shared-window address with bit 11 clear. The tables lie at multiples of 4096 from
    // the start of dynamic shared memory, which itself begins less than 2048 bytes into the window
    // (0 or the 1 KiB the system reserves); anything else must fail loudly, not decode garbage.
    if (tid == 0 && (SharedAddr(lut) & 2048u) != 0) __trap();
    const HuffLutSet* set = a.luts + im.lut_set;
    const int npairs = im.npairs;
    // per (DC, AC) table pair the two first-level tables back to back, then the second-level arena
    {
        uint4* dst = reinterpret_cast<uint4*>(lut);
        constexpr int kVecsPerTable = kFastSize * 4 / 16;
        for (int i = tid; i < npairs * 2 * kVecsPerTable; i += nth) {
            const int tsel = i / kVecsPerTable, v = i - tsel * kVecsPerTable;   // tsel = 2 * pair + is_ac
            const int tab = (tsel & 1) ? im.pair_ac[tsel >> 1] : im.pair_dc[tsel >> 1];
            dst[i] = __ldg(reinterpret_cast<const uint4*>(set->fast[tab]) + v);
        }
        uint4* sdst = dst + npairs * 2 * kVecsPerTable;
        const int nsub_vecs = int((__ldg(&set->sub_used) + 3u) >> 2);
        for (int i = tid; i < nsub_vecs; i += nth) sdst[i] = __ldg(reinterpret_cast<const uint4*>(set->sub) + i);
    }
    if (tid < 8) pair_tab[tid] = tid < 2 * npairs ? ((tid & 1) ? im.pair_ac[tid >> 1] : im.pair_dc[tid >> 1]) : 0;
    {
        const int bpm = im.bpm;
        int c = tid % bpm;
        for (int j = tid; j < K1Smem<S>::kSchedLen; j += nth) {
            sched[j] = uint16_t(SharedAddr(lut) + (uint32_t(im.mcu_pair[c]) << 12));   // the window is < 64 KiB
            c = (c + nth) % bpm;
        }
    }
    LutView lv;
    lv.fast_sa = SharedAddr(lut);
    lv.sub_sa = lv.fast_sa + uint32_t(npairs) * 4096u;
    lv.set = set;
    lv.pair_tab = pair_tab;
    return lv;
}

// One subsequence's bytes into a slot of kSlotStride words, big-endian (bit 31 of a word is the first
// bit of the stream, huff_core.cuh); the last vector's final word lies beyond the slot and is not kept.
template <int S>
__device__ __forceinline__ void StageSlotVec(uint32_t* slot, const uint8_t* src, int v) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(src) + v);
    uint32_t* w = slot + v * 4;
    w[0] = ByteSwap32(q.x); w[1] = ByteSwap32(q.y); w[2] = ByteSwap32(q.z);
    if (v != K1Smem<S>::kSlotVecs - 1) w[3] = ByteSwap32(q.w);
}

// Inline destuffing (K1Args::inline_destuff, k1_fused only): slot j receives raw bytes [j S, j S + S + 4) of the picture's
// entropy-coded data (aligned 16-byte loads shifted by raw_skip), then each thread destuffs its own slot in place by K0's
// rules (k0_core.cuh: ClassifyPiece): FF 00 -> FF, FF FF -> fill; a slot without FF stays as it is. The data end at the FF D9
// that ends the caller's buffer. Behind each slot's destuffed bytes go the picture's next destuffed bytes - the look-ahead
// of a symbol that crosses the slot's end, taken from the next slot once it is compacted, for the CTA's last slot from the
// raw bytes behind it - and zeros behind the data's end, as K0 leaves them. What only K0 handles - a marker before that
// FF D9, a picture without destuffed bytes, a slot too short to serve its neighbour's look-ahead - counts in counters[0]:
// the host then redoes the lane on K0's clean stream (Lane::Finish). me.end_bit becomes the slot's destuffed length; the
// result is where the picture's real bytes end in the slot's buffer, in bits (past its end when they do not end there).
template <int S>
__device__ __forceinline__ uint32_t StageInline(K1Smem<S>& sm, const K1Args& a, const ImageDesc& im, Sub& me) {
    constexpr int kStride = K1Smem<S>::kSlotStride, V = S / 16 + 1;
    const int tid = threadIdx.x;
    const uint8_t* const raw = a.raw + im.raw_off;   // 16-byte aligned; the data start raw_skip bytes in
    const uint32_t skip = im.raw_skip, q = skip >> 2, r = 8u * (skip & 3u), data_end = im.raw_len - 2u;
    const uint32_t st = sm.start[tid];
    const uint32_t prev = (me.active && st > 0u) ? uint32_t(__ldg(raw + skip + st - 1u)) : 0u;   // a stuffing 00 may open the slot
    for (int idx = tid; idx < T * V; idx += T) {
        const int slot = idx / V, v = idx - slot * V;
        const uint32_t so = sm.start[slot];
        if (so == ~0u) continue;
        const uint4* src = reinterpret_cast<const uint4*>(raw + so) + v;
        const uint4 x = __ldg(src), y = __ldg(src + 1);
        // words q .. q + 4 of x:y hold the vector's 16 bytes shifted by raw_skip (+ 4 bytes)
        const uint32_t w0 = q == 0u ? x.x : q == 1u ? x.y : q == 2u ? x.z : x.w;
        const uint32_t w1 = q == 0u ? x.y : q == 1u ? x.z : q == 2u ? x.w : y.x;
        uint32_t* w = sm.words + slot * kStride + v * 4;
        w[0] = ByteSwap32(__funnelshift_r(w0, w1, r));
        if (v != V - 1) {   // (the last vector: only its first word, which holds the byte after the slot)
            const uint32_t w2 = q == 0u ? x.z : q == 1u ? x.w : q == 2u ? y.x : y.y;
            const uint32_t w3 = q == 0u ? x.w : q == 1u ? y.x : q == 2u ? y.y : y.z;
            const uint32_t w4 = q == 0u ? y.x : q == 1u ? y.y : q == 2u ? y.z : y.w;
            w[1] = ByteSwap32(__funnelshift_r(w1, w2, r));
            w[2] = ByteSwap32(__funnelshift_r(w2, w3, r));
            w[3] = ByteSwap32(__funnelshift_r(w3, w4, r));
        }
    }
    __syncthreads();
    uint8_t* const b = reinterpret_cast<uint8_t*>(sm.words + tid * kStride);   // byte i of the stream at b[i ^ 3] (big-endian words)
    uint32_t c = 0;
    bool bad = false;
    if (me.active) {
        const uint32_t n = min(uint32_t(S), data_end - st);   // raw bytes of the slot before the data's end
        uint32_t i = prev == 0xFFu ? 0u : n;                  // first byte that is not kept in place
        for (int k = 0; k < S / 4 && i == n; k++) {
            if (uint32_t(4 * k) >= n) break;
            uint32_t x = sm.words[tid * kStride + k];
            if (uint32_t(4 * k + 4) > n) x &= ~(0xFFFFFFFFu >> (8u * (n - uint32_t(4 * k))));
            const uint32_t m = __vcmpeq4(x, 0xFFFFFFFFu);
            if (m) i = uint32_t(4 * k) + uint32_t(__clz(m) >> 3);
        }
        c = i;
        uint32_t p = i ? uint32_t(b[(i - 1u) ^ 3u]) : prev;
        for (; i < n; i++) {
            const uint32_t x = b[i ^ 3u];
            const uint32_t nx = i + 1u < n ? uint32_t(b[(i + 1u) ^ 3u]) : (st + n < data_end ? uint32_t(b[n ^ 3u]) : 0xFFu);
            if (x == 0xFFu && nx != 0u && nx != 0xFFu) bad = true;   // a marker before the buffer's final FF D9
            if (x != 0xFFu ? p != 0xFFu : nx == 0u) b[(c++) ^ 3u] = uint8_t(x);
            p = x;
        }
        if (c < 16u && (!me.last || c == 0u)) bad = true;
        me.end_bit = c * 8u;
    }
    sm.endbit[tid] = c * 8u;
    __syncthreads();
    uint32_t real = 0;   // bytes of the picture's data in the look-ahead
    if (me.active && tid < T - 1) {
        const uint8_t* nb = reinterpret_cast<const uint8_t*>(sm.words + (tid + 1) * kStride);
        const uint32_t cn = sm.endbit[tid + 1] >> 3, e = ((c + 3u) & ~3u) + 12u;
        for (uint32_t i = c, k = 0; i < e; i++, k++) b[i ^ 3u] = k < cn ? nb[k ^ 3u] : uint8_t(0);
        real = min(e - c, cn);
    }
    if (tid >= T - 32) {   // the last warp: the look-ahead of the CTA's last slot, from the 32 raw bytes behind it
        const uint32_t sl = sm.start[T - 1];
        if (sl != ~0u) {
            const uint32_t lane = uint32_t(tid & 31), cl = sm.endbit[T - 1] >> 3, pos = sl + S + lane;
            const uint32_t x = pos < data_end ? uint32_t(__ldg(raw + skip + pos)) : 0u;
            uint32_t nx = __shfl_down_sync(0xFFFFFFFFu, x, 1), p = __shfl_up_sync(0xFFFFFFFFu, x, 1);
            if (pos + 1u >= data_end) nx = 0xFFu;
            else if (lane == 31u) nx = __ldg(raw + skip + pos + 1u);
            if (lane == 0u) p = __ldg(raw + skip + pos - 1u);
            const bool keep = pos < data_end && (x != 0xFFu ? p != 0xFFu : nx == 0u);
            const uint32_t km = __ballot_sync(0xFFFFFFFFu, keep), at = __popc(km & ((1u << lane) - 1u)), tot = __popc(km);
            const uint32_t want = ((cl + 3u) & ~3u) + 12u - cl;
            uint8_t* lb = reinterpret_cast<uint8_t*>(sm.words + (T - 1) * kStride);
            if (keep && at < want) lb[(cl + at) ^ 3u] = uint8_t(x);
            if (lane >= tot && lane < want) lb[(cl + lane) ^ 3u] = 0;
            if (lane == 0u && tot < want && sl + S + 32u < data_end) bad = true;
            if (tid == T - 1) real = min(want, tot);
        }
    }
    if (bad) atomicAdd(&a.counters[0], 1u);
    return me.active ? 8u * (c + real) : 0u;
}

template <int S, bool INL>
__device__ __forceinline__ LutView StageCta(K1Smem<S>& sm, uint32_t* lut, const K1Args& a, const ImageDesc& im, Sub& me) {
    const int tid = threadIdx.x;
    sm.start[tid] = me.active ? uint32_t(me.start - im.data_off) : ~0u;
    const LutView lv = StageTables<S>(lut, sm.sched, sm.pair_tab, a, im);
    __syncthreads();
    uint32_t data_bits = 0;
    if (INL) {
        data_bits = StageInline<S>(sm, a, im, me);
    } else {
        constexpr int V = K1Smem<S>::kSlotVecs;
        for (int idx = tid; idx < T * V; idx += T) {
            const int slot = idx / V, v = idx - slot * V;
            const uint32_t st = sm.start[slot];
            if (st == ~0u) continue;
            StageSlotVec<S>(sm.words + slot * K1Smem<S>::kSlotStride, a.scan + im.data_off + st, v);
        }
    }
    __syncthreads();
    // (the staging offsets are not needed any more: the end of the slot's data, as 8 x the shared address of its first
    // word + 64 + its length in bits, for WriteBody's check)
    if (INL) sm.start[tid] = 8u * SharedAddr(sm.words + tid * K1Smem<S>::kSlotStride) + 64u + data_bits;
    return lv;
}

// ---------------------------------------------------------------- k1_sync
//
// A CTA owns TO = T - H consecutive subsequences of one image; its first H threads re-decode the H
// subsequences before them (the halo, owned by the previous CTA) so that the state entering the
// first owned subsequence is, almost always, already the synchronised one in round 0. Nothing the
// halo threads compute is stored; round >= 1 verifies every CTA boundary against the owner's
// result and repairs the few that differ.

// What a thread of the synchronisation pass hands to the write pass when both run in one kernel (k1_fused).
struct SyncOut {
    Sub me;             // the thread's subsequence (halo slots: as decoded, not owned)
    LutView lv;
    uint32_t img;
    uint32_t state;     // end state + block count of the subsequence
    uint32_t used;      // key of the state it was decoded from (= the predecessor's end state once synchronised)
    uint32_t nnz;       // coefficient entries it produces (padded)
    bool live;          // false: the CTA left early (round > 0, nothing to repair)
};

// FUSED: round 0 inside k1_fused - the per-round counter counts nothing here (k1_fused counts boundary mismatches itself).
template <int S, bool FUSED, bool INL>
__device__ __forceinline__ SyncOut SyncBody(const K1Args& a, K1Smem<S>& sm, uint32_t* lut, int round, int max_iters, const uint32_t cta) {
    SyncOut so;
    so.live = false;
    const int tid = threadIdx.x;
    const uint32_t img = ImageOfCta<T * K1Smem<S>::kSlotStride>(a, sm.words, cta);
    const ImageDesc& im = a.images[img];
    const int H = a.halo, TO = T - H;
    const int64_t gi = int64_t(cta) * TO + tid - H;
    const uint32_t g = uint32_t(gi);
    const bool owned = tid >= H;
    Sub me = Locate<S, INL>(a, im, gi, round > 0);
    if (round > 0 && !owned) me.active = false;   // later rounds read the owner's state instead of a halo
    if (round == 0 && owned && me.in_range) a.sub_seg[g] = me.seg;
    if (round == 0) {
        // this CTA's share of the batch's block records starts as "never decoded": blocks a damaged stream
        // does not reach, or a region of interest leaves out, then decode as zero
        const uint32_t per = (a.rec_fill_vecs + gridDim.x - 1) / gridDim.x;
        const uint32_t v0 = min(cta * per, a.rec_fill_vecs), v1 = min(v0 + per, a.rec_fill_vecs);
        uint4* dst = reinterpret_cast<uint4*>(a.blk_rec);
        for (uint32_t v = v0 + uint32_t(tid); v < v1; v += T) dst[v] = make_uint4(~0u, ~0u, ~0u, ~0u);
    }

    uint32_t my_used = 0, out = 0, old_out = kNoState;
    if (round > 0) {
        // Does any owned subsequence start from a state that is not its predecessor's end state (the CTA
        // boundary after a neighbour changed, or a chain an earlier round left unfinished)?
        int need0 = 0;
        if (me.active && !me.first) need0 = (StateKey(a.state[g - 1]) != a.used[g]);
        if (!__syncthreads_or(need0)) return so;
        if (me.active) {
            my_used = a.used[g];
            out = a.state[g];
            old_out = out;
        }
    }
    const LutView lv = StageCta<S, INL>(sm, lut, a, im, me);
    const int bpm = im.bpm;
    const uint32_t slots_sa = SharedAddr(sm.words);
    const uint32_t sched_sa = SharedAddr(sm.sched);
    auto decode = [&](uint32_t sub, uint32_t key) {   // result state returned, entry count left in sm.nnz[sub]
        uint32_t n;
        const uint32_t st = DecodeCount(slots_sa + sub * uint32_t(K1Smem<S>::kSlotStride * 4), lv, sched_sa, bpm, key, sm.endbit[sub], &n);
        sm.nnz[sub] = n;
        return st;
    };

    uint32_t ndecodes = 0;
    sm.endbit[tid] = me.end_bit;
    sm.nnz[tid] = (round > 0 && me.active) ? a.nnz[g] : 0u;
    if (tid == 0) sm.scratch[0] = 0;   // work-queue length
    __syncthreads();
    if (round == 0 && me.active) {
        // guess for a mid-segment start: aligned on a symbol, first block of an MCU, DC next
        my_used = 0;
        out = decode(uint32_t(tid), 0);
        ndecodes++;
    }
    sm.state[tid] = out;
    sm.used[tid] = my_used;
    // state entering the first active thread (later rounds: snapshot of the owner's result; the
    // neighbouring CTA may still be changing it — a change is caught by the boundary counter and the
    // next round)
    uint32_t in0 = my_used;
    if (round > 0 && tid == H && me.active && !me.first) in0 = StateKey(a.state[g - 1]);
    const bool has_pred = (round == 0) ? (tid > 0) : (tid > H);
    const bool can_redo = me.active && !me.first;
    const int lane = tid & 31;
    // CTA-local fix-up: re-decode while the predecessor's end state is not the state used. The
    // subsequences that need it are compacted into a queue so that the re-decodes occupy as few
    // warps as possible (a warp with one busy lane costs as many issue slots as a full one).
    for (int iter = 0; iter < max_iters; iter++) {
        __syncthreads();
        // a predecessor slot that maps to no data (before the image's first subsequence) hands over
        // nothing: such a thread is `first` and never re-decodes, so the value read is irrelevant
        const uint32_t in = has_pred ? StateKey(sm.state[tid - 1]) : in0;
        const bool need = can_redo && in != sm.used[tid];
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, need);
        uint32_t base = 0;
        if (lane == 0 && mask) base = atomicAdd(&sm.scratch[0], uint32_t(__popc(mask)));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (need) sm.queue[base + __popc(mask & ((1u << lane) - 1u))] = (in << 16) | uint32_t(tid);
        __syncthreads();
        const uint32_t n = sm.scratch[0];
        if (n == 0) break;
        uint32_t item = 0, res = 0;
        if (uint32_t(tid) < n) {
            item = sm.queue[tid];
            res = decode(item & 0xFFFFu, item >> 16);
            ndecodes++;
        }
        __syncthreads();
        if (uint32_t(tid) < n) {
            sm.state[item & 0xFFFFu] = res;
            sm.used[item & 0xFFFFu] = item >> 16;
        }
        if (tid == 0) sm.scratch[0] = 0;
    }
    __syncthreads();
    out = sm.state[tid];
    my_used = sm.used[tid];
    const uint32_t my_nnz = sm.nnz[tid];
    const bool mine = owned && me.active;
    if (mine) {
        a.state[g] = out;
        a.used[g] = my_used;
        a.nnz[g] = my_nnz;
    }
    // A change of the state handed to the next CTA means that CTA must look again.
    const bool hands_over = mine && !me.last && (tid == T - 1);
    if (!FUSED && hands_over && (old_out == kNoState || StateKey(old_out) != StateKey(out))) atomicAdd(&a.counters[round], 1u);
    if (ndecodes) atomicAdd(&a.counters[kMaxSyncRounds + round], ndecodes);

    // CTA partial for the block-position scan: (contains a segment start, blocks after the last start)
    uint32_t* red = sm.scratch;
    if (tid == 0) { red[0] = 0; red[1] = 0; }
    __syncthreads();
    if (mine && me.first) atomicMax(&red[0], uint32_t(tid) + 1u);
    __syncthreads();
    const uint32_t last_first = red[0];   // 0 = none, else tid + 1
    if (mine && (last_first == 0 || uint32_t(tid) + 1u >= last_first)) atomicAdd(&red[1], StateBlocks(out));
    __syncthreads();
    if (tid == 0) a.cta_partial[cta] = make_uint2(last_first != 0 ? 1u : 0u, red[1]);
    // entries produced by the CTA (plain sum: entry offsets run through the whole image)
    if (tid == 0) red[2] = 0;
    __syncthreads();
    if (mine && my_nnz) atomicAdd(&red[2], my_nnz);
    __syncthreads();
    if (tid == 0) a.cta_entries[cta] = red[2];
    so.me = me;
    so.lv = lv;
    so.img = img;
    so.state = out;
    so.used = my_used;
    so.nnz = my_nnz;
    so.live = true;
    return so;
}

template <int S>
__global__ void __launch_bounds__(T) k1_sync(K1Args a, int round, int max_iters) {
    PdlEntry();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* const lut = reinterpret_cast<uint32_t*>(smem_raw);
    K1Smem<S>& sm = *reinterpret_cast<K1Smem<S>*>(smem_raw + a.lut_smem_bytes);
    (void)SyncBody<S, false, false>(a, sm, lut, round, max_iters, blockIdx.x);
}

// ---------------------------------------------------------------- k1_scan
//
// One CTA per image: exclusive scan over the image's CTA partials, kScanThreads at a time. Block
// positions are a segmented sum (a CTA holding a restart-interval start cuts the chain: its
// partial already counts only the blocks after its last start), entry offsets a plain sum.
constexpr int kScanThreads = 256;

__global__ void __launch_bounds__(kScanThreads) k1_scan(K1Args a) {
    PdlEntry();
    __shared__ uint32_t s_v[kScanThreads / 32], s_f[kScanThreads / 32], s_e[kScanThreads / 32];
    const uint32_t img = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t c0 = a.img_cta0[img], c1 = a.img_cta0[img + 1];
    uint32_t carry_b = 0, carry_e = 0;   // what enters the current chunk (same in every thread)
    for (uint32_t base = c0; base < c1; base += kScanThreads) {
        const uint32_t k = base + tid;
        uint2 part = make_uint2(0u, 0u);
        uint32_t ents = 0;
        if (k < c1) {
            part = a.cta_partial[k];
            ents = a.cta_entries[k];
        }
        uint32_t f = part.x ? 1u : 0u, v = part.y, e = ents;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t pv = __shfl_up_sync(0xFFFFFFFFu, v, d);
            const uint32_t pf = __shfl_up_sync(0xFFFFFFFFu, f, d);
            const uint32_t pe = __shfl_up_sync(0xFFFFFFFFu, e, d);
            if (lane >= d) {
                if (!f) v += pv;
                f |= pf;
                e += pe;
            }
        }
        __syncthreads();   // previous iteration's readers are done
        if (lane == 31) { s_v[warp] = v; s_f[warp] = f; s_e[warp] = e; }
        __syncthreads();
        // what precedes this warp inside the chunk, then the chunk's own carry
        uint32_t pre_v = 0, pre_f = 0, pre_e = 0;
        for (int w = 0; w < warp; w++) {
            pre_v = s_f[w] ? s_v[w] : pre_v + s_v[w];
            pre_f |= s_f[w];
            pre_e += s_e[w];
        }
        if (!pre_f) pre_v += carry_b;
        pre_e += carry_e;
        // inclusive -> exclusive inside the warp
        uint32_t xv = __shfl_up_sync(0xFFFFFFFFu, v, 1), xf = __shfl_up_sync(0xFFFFFFFFu, f, 1), xe = __shfl_up_sync(0xFFFFFFFFu, e, 1);
        if (lane == 0) { xv = 0; xf = 0; xe = 0; }
        if (k < c1) a.cta_carry[k] = make_uint2(xf ? xv : xv + pre_v, xe + pre_e);
        // carry into the next chunk = inclusive value at the chunk's last element
        uint32_t tot_v = 0, tot_f = 0, tot_e = 0;
        for (int w = 0; w < kScanThreads / 32; w++) {
            tot_v = s_f[w] ? s_v[w] : tot_v + s_v[w];
            tot_f |= s_f[w];
            tot_e += s_e[w];
        }
        carry_b = tot_f ? tot_v : tot_v + carry_b;
        carry_e += tot_e;
    }
}

// ---------------------------------------------------------------- k1_write

// k1_fused's DC integration splits a picture's blocks among its CTAs at the block each CTA's first own subsequence starts
// in: the block in progress there for a subsequence inside a restart interval (`excl` = blocks the interval ended
// before it), the interval's end for one behind the interval's data, the picture's end for one behind the picture.
// Clamped so that the split points never decrease, whatever a damaged stream made of the counts.
constexpr int kDcPosSlot = 32;   // K1Smem::scratch words holding the range (IntegrateDc)
template <bool INL>
__device__ __forceinline__ uint32_t BlockPos(const K1Args& a, const ImageDesc& im, const Sub& s, uint32_t excl) {
    if (!s.in_range) return im.nblocks;
    const SegmentDesc sd = SegmentOf<INL>(a, im, s.seg);
    const uint32_t p = sd.blk_first + (!s.active ? sd.blk_count : s.first ? 0u : min(excl, sd.blk_count));
    return min(p, im.nblocks);
}

// The write pass behind the staging: `st`, `my_nnz`, `key` = the thread's synchronised end state, entry count and start
// state. FUSED (k1_fused): the same CTA has just synchronised - what enters it from the picture's earlier CTAs is read
// from their partials as soon as each has published them (`cta_flag`), and the state handed over at the CTA boundary is
// checked against the owner's.
template <int S, bool FUSED, bool INL>
__device__ __forceinline__ void WriteBody(const K1Args& a, K1Smem<S>& sm, const LutView& lv, uint32_t img, const ImageDesc& im, const Sub& me,
                                          uint32_t st, uint32_t my_nnz, uint32_t key, const uint32_t cta) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (cta == 0 && tid < 64) a.counters_next[tid] = 0;   // the next batch's counters (this batch's are read back after K3)
    const uint32_t nb = StateBlocks(st);
    // Two scans over the CTA: block positions (segmented: a segment start resets the count) and
    // entry offsets (plain, they run through the whole image).
    uint32_t v = nb, e = my_nnz;
    uint32_t f = (me.active && me.first) ? 1u : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t pv = __shfl_up_sync(0xFFFFFFFFu, v, d);
        const uint32_t pf = __shfl_up_sync(0xFFFFFFFFu, f, d);
        const uint32_t pe = __shfl_up_sync(0xFFFFFFFFu, e, d);
        if (lane >= d) {
            if (!f) v += pv;
            f |= pf;
            e += pe;
        }
    }
    constexpr int kW = T / 32;
    static_assert(3 * kW + 2 <= 40, "scratch");
    uint32_t* wsum = sm.scratch;               // [kW] warp totals (value of the open segment at warp end)
    uint32_t* wflag = sm.scratch + kW;         // [kW] warp contains a start
    uint32_t* wents = sm.scratch + 2 * kW;     // [kW] warp entry totals
    uint32_t* carry_s = sm.scratch + 3 * kW;   // [2] what enters the CTA: blocks, entries
    if (lane == 31) { wsum[warp] = v; wflag[warp] = f; wents[warp] = e; }
    // what enters this CTA from the previous CTAs of the image: k1_scan prepared it (a look-back here
    // would re-read every earlier partial of the image, quadratic for the 8192x8192 pictures)
    if (FUSED) {
        // One lane per earlier CTA of the picture, 32 at a time from the nearest backwards, each read as soon as its owner has
        // published it (a lower CTA index: dispatched before this one, and it never waits for a later one). Entries: plain sum.
        // Blocks: the partials from the last CTA holding a restart-interval start on (its partial counts only the blocks
        // after that start).
        if (warp == 0) {
            const int64_t first = int64_t(__ldg(a.img_cta0 + img));
            uint32_t cb = 0, ents = 0;
            bool open = true;
            for (int64_t hi = int64_t(cta); hi > first; hi -= 32) {
                const int64_t k = hi - 32 + lane;   // lane 31: the CTA just before the ones already summed
                uint2 part = make_uint2(0u, 0u);
                if (k >= first) {
                    uint32_t f;
                    do {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(f) : "l"(a.cta_flag + k) : "memory");
                    } while (f == 0u);
                    part = __ldcg(a.cta_partial + k);
                    ents += __ldcg(a.cta_entries + k);
                }
                if (open) {
                    const uint32_t starts = __ballot_sync(0xFFFFFFFFu, part.x != 0);
                    const int from = starts ? 31 - __clz(starts) : 0;
                    if (lane >= from) cb += part.y;
                    open = starts == 0u;
                }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                cb += __shfl_xor_sync(0xFFFFFFFFu, cb, d);
                ents += __shfl_xor_sync(0xFFFFFFFFu, ents, d);
            }
            if (lane == 0) {
                carry_s[0] = cb;
                carry_s[1] = ents;
            }
        }
    } else if (tid == 0) {
        const uint2 cin = a.cta_carry[cta];
        carry_s[0] = cin.x;
        carry_s[1] = cin.y;
    }
    __syncthreads();
    if (tid == 0) {   // statistics: coefficient entries the batch writes (pads included), read back with the round counters
        uint32_t t = 0;
        for (int w = 0; w < kW; w++) t += wents[w];
        if (t) atomicAdd(&a.counters[2 * kMaxSyncRounds], t);
    }
    uint32_t add = 0, eadd = carry_s[1];
    bool open = (f == 0);   // no segment start at or before this thread inside its warp
    for (int w = warp - 1; w >= 0; w--) {
        eadd += wents[w];
        if (open) {
            add += wsum[w];
            if (wflag[w]) open = false;
        }
    }
    if (open) add += carry_s[0];
    const uint32_t excl = (me.active && me.first) ? 0u : v + add - nb;
    uint32_t n = e + eadd - my_nnz;   // this thread's first entry, relative to the image

    if (!me.active) return;
    // ---- final decode: every symbol with magnitude bits becomes one 32-bit entry of the
    // image's coefficient stream, written at its final position (each thread owns a contiguous
    // run of the stream, eight entries per 256-bit store); every block end records the index one
    // past the block's last entry, every DC symbol its difference in the compact per-block array.
    // A block's entries begin where the previous block's end (block 0: entry 0): what lies between
    // two threads' runs or two restart intervals is zero padding (position 0, which K2 overwrites
    // with the DC). No clearing, no read-modify-write, no ownership hand-over: a thread decodes
    // exactly the symbols that start inside its subsequence, as in the counting passes.
    const SegmentDesc sd = SegmentOf<INL>(a, im, me.seg);
    const uint32_t blk0 = sd.blk_first + excl, limit = sd.blk_first + sd.blk_count;
    // running pointers: the current block's record {end-of-entries index, DC} and the next 32-byte
    // entry group of this thread's run; the run never leaves its reservation [n, n_end), the
    // reservations never leave the image's arena
    BlockRec* recs = a.blk_rec + im.blk0;
    BlockRec* rp = recs + blk0;
    const uint32_t rp_stop = uint32_t(reinterpret_cast<uintptr_t>(recs + limit));   // low word is enough: < 4 GiB of records
    uint32_t* ep = a.entries + im.ent0 + n;
    const uint32_t n_end = min(n + my_nnz, im.ent_cap & ~7u);
    Lane ln;
    ln.Init(SharedAddr(sm.words + tid * K1Smem<S>::kSlotStride), SharedAddr(sm.sched), key, me.end_bit);
    // The last four entries (oldest in q0) and, once four have gathered, the first half of the group of
    // eight (h0..h3): a group leaves as ONE 256-bit store, a whole 32-byte sector. The store path is the
    // write pass's second bottleneck (every lane writes its own run, so a store instruction is as many
    // transactions as it has active lanes): half the stores of the 128-bit form (profiles/r01g_*).
    uint32_t q0 = 0, q1 = 0, q2 = 0, q3 = 0, h0 = 0, h1 = 0, h2 = 0, h3 = 0;
    int dcv = 0;                               // DC difference of the block in progress, when its DC symbol was ours
    uint32_t has_dc = StateZ(key) == 0 ? 1u : 0u;
    if (blk0 < limit && me.end_bit != 0) {
        for (;;) {
            const uint32_t win = ln.Peek();
            uint32_t en = ln.Lookup(win);
            if (IsLink(en)) en = ResolveLink(lv, en, ln.off, win);
            const uint32_t nxt = ln.acc + en;
            // RECEIVE + EXTEND (T.81 F.2.2.1) on the magnitude bits that follow the code; the DC
            // difference goes to the block's record, every symbol with magnitude bits becomes an entry
            // whose upper half is the zig-zag index AFTER the symbol (+ state bits K2 masks off)
            asm volatile(
                "{\n\t"
                ".reg .pred pdc, pnz, pneg, pfl, pst, phalf;\n\t"
                ".reg .b32 sz, bits, sh, t, rs, ex, m, v, zq;\n\t"
                "shr.u32 sz, %11, 28;\n\t"
                "and.b32 bits, %11, 31;\n\t"
                "sub.u32 sh, bits, sz;\n\t"
                "shl.b32 t, %12, sh;\n\t"
                "sub.u32 rs, 32, sz;\n\t"
                "shf.r.clamp.b32 ex, t, 0, rs;\n\t"
                "bmsk.clamp.b32 m, 0, sz;\n\t"
                "setp.lt.s32 pneg, t, 0;\n\t"
                "selp.b32 m, 0, m, pneg;\n\t"
                "sub.s32 v, ex, m;\n\t"
                "and.b32 zq, %13, 0x7e00000;\n\t"
                "setp.eq.u32 pdc, zq, 0;\n\t"
                "@pdc mov.b32 %6, v;\n\t"
                "setp.ne.u32 pnz, sz, 0;\n\t"
                "shr.u32 zq, %14, 21;\n\t"
                "@pnz mov.b32 %0, %1;\n\t"
                "@pnz mov.b32 %1, %2;\n\t"
                "@pnz mov.b32 %2, %3;\n\t"
                "@pnz prmt.b32 %3, v, zq, 0x5410;\n\t"
                "@pnz add.u32 %4, %4, 1;\n\t"
                "and.b32 zq, %4, 7;\n\t"
                "setp.eq.and.u32 phalf, zq, 4, pnz;\n\t"
                "setp.eq.and.u32 pfl, zq, 0, pnz;\n\t"
                "@phalf mov.b32 %7, %0;\n\t"
                "@phalf mov.b32 %8, %1;\n\t"
                "@phalf mov.b32 %9, %2;\n\t"
                "@phalf mov.b32 %10, %3;\n\t"
                "setp.le.and.u32 pst, %4, %15, pfl;\n\t"
                "@pst st.global.v8.b32 [%5], {%7, %8, %9, %10, %0, %1, %2, %3};\n\t"
                "@pfl add.u64 %5, %5, 32;\n\t"
                "}"
                : "+r"(q0), "+r"(q1), "+r"(q2), "+r"(q3), "+r"(n), "+l"(ep), "+r"(dcv), "+r"(h0), "+r"(h1), "+r"(h2), "+r"(h3)
                : "r"(en), "r"(win), "r"(ln.acc), "r"(nxt), "r"(n_end)
                : "memory");
            ln.CommitWrite(nxt, rp, n, rp_stop, dcv, has_dc);
            if (ln.acc & kAccStop) break;
        }
        // Inline destuffing: the symbol that ended the picture's last block must end inside the picture's data. Behind
        // them a thread reads zeros, and how many zero bits it reads before it stops depends on the layout (K0's decode
        // of the same bytes may come out short where this one did not): counters[0], the host redoes the lane on K0's
        // stream. A complete scan ends its last block inside its data.
        // (the read position is 8 wp + (acc & 31) - 64 bits from the slot's start: wp is the address of the word after the
        // next; sm.start holds the end of the data in the same terms, StageCta)
        if (INL && uint32_t(reinterpret_cast<uintptr_t>(rp)) == rp_stop && (ln.wp << 3) + (ln.acc & 31u) > sm.start[tid])
            atomicAdd(&a.counters[0], 1u);
    }
    // per-image status (read back by the host with the round counters): the interval ran out of bytes before its last
    // block (truncated or damaged scan)
    // (inline destuffing: what the decode found past the data's end depends on the subsequence layout - the host redoes the
    // picture on K0's layout, counters[0])
    if (me.last && blk0 < limit && uint32_t(rp - recs) < limit) {
        atomicOr(&a.status[img].flags, kDecodeShort);
        if (INL) atomicAdd(&a.counters[0], 1u);
    }
    // a block still in progress whose DC symbol was ours: the thread that ends it stores only the end index
    if (has_dc && (ln.acc & kAccZMask) != 0 && blk0 < limit && me.end_bit != 0) rp->dc = int16_t(dcv);
    if (n & 7u) {   // last, partial group: padded with entries for position 0, which K2 overwrites with the DC anyway
        for (; n & 7u; n++) {
            q0 = q1; q1 = q2; q2 = q3; q3 = kPadEntry;
            if ((n & 7u) == 3u) { h0 = q0; h1 = q1; h2 = q2; h3 = q3; }   // this entry completed the first half
        }
        if (n <= n_end) {
            reinterpret_cast<uint4*>(ep)[0] = make_uint4(h0, h1, h2, h3);
            reinterpret_cast<uint4*>(ep)[1] = make_uint4(q0, q1, q2, q3);
        }
        ep += 8;
    }
    // groups the counting pass reserved but this pass did not fill (symbols it saw in the padding
    // after a restart interval's last block): pad them, the next block's range starts behind them
    for (; n < n_end; n += 8, ep += 8) {
        reinterpret_cast<uint4*>(ep)[0] = make_uint4(kPadEntry, kPadEntry, kPadEntry, kPadEntry);
        reinterpret_cast<uint4*>(ep)[1] = make_uint4(kPadEntry, kPadEntry, kPadEntry, kPadEntry);
    }
}

template <int S>
__global__ void __launch_bounds__(T) k1_write(K1Args a) {
    PdlEntry();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* const lut = reinterpret_cast<uint32_t*>(smem_raw);
    K1Smem<S>& sm = *reinterpret_cast<K1Smem<S>*>(smem_raw + a.lut_smem_bytes);
    const int tid = threadIdx.x;
    const uint32_t cta = blockIdx.x;
    const uint32_t img = ImageOfCta<T * K1Smem<S>::kSlotStride>(a, sm.words, cta);
    const ImageDesc& im = a.images[img];
    const int H = a.halo, TO = T - H;
    const int64_t gi = int64_t(cta) * TO + tid - H;
    const uint32_t g = uint32_t(gi);
    Sub me = Locate<S, false>(a, im, gi, true);
    if (tid < H) me.active = false;   // halo slots belong to the previous CTA
    const LutView lv = StageCta<S, false>(sm, lut, a, im, me);
    const uint32_t st = me.active ? a.state[g] : 0;
    const uint32_t my_nnz = me.active ? a.nnz[g] : 0;
    uint32_t key = 0;
    if (me.active && !me.first) key = StateKey(a.state[g - 1]);
    WriteBody<S, false, false>(a, sm, lv, img, im, me, st, my_nnz, key, cta);
}

// ---------------------------------------------------------------- k1_fused
//
// Counting and write pass in ONE kernel for pictures of up to 256 K1 CTAs (4 MB of scan at 128-byte subsequences): a CTA
// synchronises its subsequences exactly as round 0 of k1_sync does, publishes its block / entry counts and the state
// it hands over, and goes straight on to write - the bytes and the tables are still in shared memory (the second
// staging, a launch and its tail are saved), and while one picture's CTAs walk their chains the others' already
// write. What the verifying round of k1_sync checks is checked here by the CTA itself: the state its halo threads
// derived for its first subsequence must be the one the owner (the CTA before it) ended on; every mismatch is counted
// in counters[0], and the host then falls back to the separate kernels for the batch (none on the benchmark batches,
// forced in tests with ROCJPEG_B200_HALO=1). With K1Args::k1_dc the CTA then turns the DC differences of its share of the
// picture's blocks into absolute DC values (IntegrateDc), and no DC kernel follows.
template <int S, bool INL>
__device__ void IntegrateDc(const K1Args& a, uint32_t* scratch, uint32_t img, uint32_t cta);

// (the register cap replaces __launch_bounds__(T), which cannot be combined with it: the DC integration behind the write
// loop would otherwise raise the kernel from the decode loops' 46 registers to 48)
template <int S, bool INL>
__global__ void __maxnreg__(46) k1_fused(K1Args a, int max_iters) {
    PdlEntry();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint32_t* const lut = reinterpret_cast<uint32_t*>(smem_raw);
    K1Smem<S>& sm = *reinterpret_cast<K1Smem<S>*>(smem_raw + a.lut_smem_bytes);
    const int tid = threadIdx.x;
    // Which CTA's work this is: a ticket, not blockIdx - the waits below are for lower indices, and a ticket holder
    // knows that every lower ticket has been drawn by a CTA that is running (whatever order the grid is dispatched in).
    __shared__ uint32_t s_ticket, s_img;
    if (tid == 0) s_ticket = atomicAdd(a.cta_flag + a.total_ctas, 1u);
    __syncthreads();
    const uint32_t cta = s_ticket;
    SyncOut so = SyncBody<S, true, INL>(a, sm, lut, 0, max_iters, cta);
    // inline destuffing, no K0 ran: the picture's first CTA writes its status - a restart interval that ends at the FF D9
    // closing the buffer - before any CTA of the picture may OR into it (they all wait for its flag below first)
    if (INL && tid == 0 && cta == __ldg(a.img_cta0 + so.img))
        a.status[so.img] = ScanStatus{1u, a.images[so.img].raw_len - 2u, 0u, 0u};
    if (tid == 0) s_img = so.img;
    // this CTA's counts and states are in global memory: let the picture's later CTAs see them
    __threadfence();
    __syncthreads();
    if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(a.cta_flag + cta), "r"(1u) : "memory");
    const int H = a.halo;
    const ImageDesc& im = a.images[so.img];
    // the state entering the CTA's first own subsequence came from the halo: is it what the owner ended on?
    if (tid == H && so.me.active && !so.me.first && cta > 0) {
        uint32_t f;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(f) : "l"(a.cta_flag + cta - 1) : "memory");
        } while (f == 0u);
        const uint32_t g = uint32_t(int64_t(cta) * (T - H));
        if (StateKey(__ldcg(a.state + g - 1)) != so.used) atomicAdd(&a.counters[0], 1u);
    }
    Sub me = so.me;
    if (tid < H) me.active = false;   // halo slots belong to the previous CTA
    WriteBody<S, true, INL>(a, sm, so.lv, so.img, im, me, me.active ? so.state : 0u, me.active ? so.nnz : 0u, so.used, cta);
    if (a.k1_dc) {
        // (ticket and picture re-read from shared memory: kept in registers across the write loop they cost two)
        const uint32_t c = *static_cast<volatile uint32_t*>(&s_ticket);
        // this CTA's records are written: the next CTA may read the DC difference its first block got from here
        __threadfence();
        __syncthreads();
        if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(a.cta_flag + c), "r"(2u) : "memory");
        IntegrateDc<S, INL>(a, sm.scratch, *static_cast<volatile uint32_t*>(&s_img), c);
    }
}

// ---------------------------------------------------------------- DC prediction

// DC difference of a block; 0 for a block no thread reached (damaged stream: the record still
// holds the 0xFF fill)
__device__ __forceinline__ int RecDc(const BlockRec& r) { return r.end == kNoEntry ? 0 : int(r.dc); }

// The DC differences of one MCU in registers (fully unrolled over the ten blocks an MCU can have, 8-byte
// loads, selects by component instead of indexing: the scalar form kept its arrays in local memory) and
// their sums per component. (A warp-cooperative variant - the 32 MCUs' records read and written as one
// coalesced run and transposed through shared memory - was measured 10-15 % slower: these kernels are bound
// by their instruction count, not by memory transactions.)
struct McuDc {
    int d[kMaxBlocksPerMcu];
    int s0, s1, s2;
    // N = unroll bound >= bpm (these kernels are bound by their instruction count: a grey picture, one block
    // per MCU, must not pay for ten predicated steps)
    template <int N>
    __device__ __forceinline__ void LoadN(const BlockRec* rec, int bpm, uint32_t comp_bits, bool active) {
        s0 = s1 = s2 = 0;
#pragma unroll
        for (int k = 0; k < N; k++) {
            d[k] = 0;
            if (active && k < bpm) {
                const uint2 r = *reinterpret_cast<const uint2*>(rec + k);
                d[k] = r.x == kNoEntry ? 0 : int(int16_t(r.y & 0xFFFFu));   // a block no thread reached counts as 0
            }
            const uint32_t comp = (comp_bits >> (2 * k)) & 3u;
            s0 += comp == 0u ? d[k] : 0;
            s1 += comp == 1u ? d[k] : 0;
            s2 += comp == 2u ? d[k] : 0;
        }
    }
    template <int N>
    __device__ __forceinline__ void StoreN(BlockRec* rec, int bpm, uint32_t comp_bits, int p0, int p1, int p2) const {
#pragma unroll
        for (int k = 0; k < N; k++) {
            const uint32_t comp = (comp_bits >> (2 * k)) & 3u;
            p0 += comp == 0u ? d[k] : 0;
            p1 += comp == 1u ? d[k] : 0;
            p2 += comp == 2u ? d[k] : 0;
            if (k < bpm) rec[k].dc = int16_t(comp == 0u ? p0 : comp == 1u ? p1 : p2);
        }
    }
    // bpm is uniform over the CTA (one picture): 1 grey, 3 4:4:4, 4 4:2:2 / 4:4:0, 6 4:2:0, up to 10 otherwise
    __device__ __forceinline__ void Load(const BlockRec* rec, int bpm, uint32_t comp_bits, bool active) {
        if (bpm == 1) LoadN<1>(rec, bpm, comp_bits, active);
        else if (bpm <= 4) LoadN<4>(rec, bpm, comp_bits, active);
        else if (bpm <= 6) LoadN<6>(rec, bpm, comp_bits, active);
        else LoadN<kMaxBlocksPerMcu>(rec, bpm, comp_bits, active);
    }
    // the integrated DC replaces the difference in every block's record; p0..p2 = predictors entering the MCU
    __device__ __forceinline__ void Store(BlockRec* rec, int bpm, uint32_t comp_bits, int p0, int p1, int p2) const {
        if (bpm == 1) StoreN<1>(rec, bpm, comp_bits, p0, p1, p2);
        else if (bpm <= 4) StoreN<4>(rec, bpm, comp_bits, p0, p1, p2);
        else if (bpm <= 6) StoreN<6>(rec, bpm, comp_bits, p0, p1, p2);
        else StoreN<kMaxBlocksPerMcu>(rec, bpm, comp_bits, p0, p1, p2);
    }
};
__device__ __forceinline__ bool ResetAt(uint32_t m, int ri) { return ri > 0 ? (m % uint32_t(ri)) == 0u : m == 0u; }

// Does MCU range [m0, m1) of an image contain a predictor reset? Returns the last one, or -1.
__device__ __forceinline__ int64_t LastReset(int64_t m0, int64_t m1, int ri) {
    if (m1 <= m0) return -1;
    if (ri <= 0) return m0 == 0 ? 0 : -1;
    const int64_t last = ((m1 - 1) / ri) * ri;
    return last >= m0 ? last : -1;
}

// RecDc through L2: the first block of a range may have got its DC difference from another SM
__device__ __forceinline__ int LoadDc(const BlockRec* r) {
    const uint2 v = __ldcg(reinterpret_cast<const uint2*>(r));
    return v.x == kNoEntry ? 0 : int(int16_t(v.y & 0xFFFFu));
}

// k1_fused, after its write pass: the DC differences of blocks [lo, hi) of the picture (BlockPos) become absolute DC values,
// the arithmetic of dc_sums / dc_apply on a range that need not start on an MCU. Every record of the range is final once
// this CTA and the one before it have written theirs: the first block's DC symbol may lie in the previous CTA, every other symbol of the
// range lies in this one. Each thread sums a contiguous run; a CTA-wide segmented scan and a decoupled look-back over the
// picture's earlier CTAs (their per-component sums after the last predictor reset, or the predictors leaving them once
// known) give the predictors entering each run. Every wait is for a lower ticket, i.e. for a running CTA that itself
// waits only for lower tickets.
template <int S, bool INL>
__device__ void IntegrateDc(const K1Args& a, uint32_t* scratch, uint32_t img, uint32_t cta) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kW = T / 32;
    const ImageDesc& im = a.images[img];
    const uint32_t first = __ldg(a.img_cta0 + img);
    uint32_t* const dc_flag = a.cta_flag + a.total_ctas + 1;
    const int H = a.halo;
    if (tid == H || tid == T - 1) {   // the range: where the CTA's first own subsequence starts, and where the next CTA's does
        // blocks entering the CTA from its restart interval (WriteBody left them in scratch) and, from the CTA's own partial,
        // those leaving it
        const uint32_t enter = scratch[3 * kW];
        const int64_t gi = int64_t(cta) * (T - H) + tid - H;
        if (tid == H) {
            scratch[kDcPosSlot] = BlockPos<INL>(a, im, Locate<S, INL>(a, im, gi, false), enter);
        } else {
            const uint2 part = a.cta_partial[cta];
            scratch[kDcPosSlot + 1] = BlockPos<INL>(a, im, Locate<S, INL>(a, im, gi + 1, false), part.y + (part.x ? 0u : enter));
        }
    }
    if (tid == 0 && cta != first) {
        uint32_t f;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(f) : "l"(a.cta_flag + cta - 1) : "memory");
        } while (f != 2u);
    }
    __syncthreads();
    const uint32_t lo = cta == first ? 0u : scratch[kDcPosSlot];
    const uint32_t hi = max(lo, scratch[kDcPosSlot + 1]);
    const uint32_t per = (hi - lo + T - 1) / T;
    const uint32_t b0 = min(lo + uint32_t(tid) * per, hi), b1 = min(b0 + per, hi);
    BlockRec* const rec = a.blk_rec + im.blk0;
    const uint32_t bpm = uint32_t(im.bpm), comp_bits = im.comp_bits;
    const int ri = im.restart_interval;
    // the run's sums after its last reset (f: it holds one)
    int s0 = 0, s1 = 0, s2 = 0;
    uint32_t f = 0;
    {
        uint32_t m = b0 / bpm, k = b0 - m * bpm;
        for (uint32_t b = b0; b < b1; b++) {
            if (k == 0 && ResetAt(m, ri)) { s0 = s1 = s2 = 0; f = 1; }
            const int d = LoadDc(rec + b);
            const uint32_t comp = (comp_bits >> (2 * k)) & 3u;
            s0 += comp == 0u ? d : 0;
            s1 += comp == 1u ? d : 0;
            s2 += comp == 2u ? d : 0;
            if (++k == bpm) { k = 0; m++; }
        }
    }
    int v0 = s0, v1 = s1, v2 = s2;
    uint32_t g = f;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int p0 = __shfl_up_sync(0xFFFFFFFFu, v0, d);
        const int p1 = __shfl_up_sync(0xFFFFFFFFu, v1, d);
        const int p2 = __shfl_up_sync(0xFFFFFFFFu, v2, d);
        const uint32_t pg = __shfl_up_sync(0xFFFFFFFFu, g, d);
        if (lane >= d) {
            if (!g) { v0 += p0; v1 += p1; v2 += p2; }
            g |= pg;
        }
    }
    int* const ws = reinterpret_cast<int*>(scratch);   // [4 w + c]: warp w's inclusive sums, [4 w + 3]: it holds a reset
    int* const carry = ws + 4 * kW;                      // predictors entering the CTA
    if (lane == 31) { ws[4 * warp] = v0; ws[4 * warp + 1] = v1; ws[4 * warp + 2] = v2; ws[4 * warp + 3] = int(g); }
    __syncthreads();
    if (warp == 0) {
        int t0 = 0, t1 = 0, t2 = 0, tf = 0;   // the CTA's own sums after its last reset
        for (int w = 0; w < kW; w++) {
            if (ws[4 * w + 3]) { t0 = ws[4 * w]; t1 = ws[4 * w + 1]; t2 = ws[4 * w + 2]; tf = 1; }
            else { t0 += ws[4 * w]; t1 += ws[4 * w + 1]; t2 += ws[4 * w + 2]; }
        }
        if (lane == 0) {
            a.cta_dc[2 * cta] = make_int4(t0, t1, t2, tf);
            __threadfence();
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(dc_flag + cta), "r"(1u) : "memory");
        }
        // one lane per earlier CTA of the picture, 32 at a time from the nearest backwards, up to the nearest one whose
        // outgoing predictors are known or whose range holds a reset
        int c0 = 0, c1 = 0, c2 = 0;
        for (int64_t top = int64_t(cta); top > int64_t(first); top -= 32) {
            const int64_t k = top - 32 + lane;
            int4 e = make_int4(0, 0, 0, 0);
            uint32_t fl = 0;
            if (k >= int64_t(first)) {
                do {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(fl) : "l"(dc_flag + k) : "memory");
                } while (fl == 0u);
                e = __ldcg(a.cta_dc + 2 * k + (fl == 2u ? 1 : 0));
            }
            const uint32_t stop = __ballot_sync(0xFFFFFFFFu, fl == 2u || e.w != 0);
            const int from = stop ? 31 - __clz(stop) : 0;
            if (lane >= from) { c0 += e.x; c1 += e.y; c2 += e.z; }
            if (stop) break;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, d);
            c1 += __shfl_xor_sync(0xFFFFFFFFu, c1, d);
            c2 += __shfl_xor_sync(0xFFFFFFFFu, c2, d);
        }
        if (lane == 0) {
            carry[0] = c0; carry[1] = c1; carry[2] = c2;
            a.cta_dc[2 * cta + 1] = tf ? make_int4(t0, t1, t2, 0) : make_int4(c0 + t0, c1 + t1, c2 + t2, 0);
            __threadfence();
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(dc_flag + cta), "r"(2u) : "memory");
        }
    }
    __syncthreads();
    // predictors entering the run: the warp's exclusive prefix, the earlier warps' sums back to the last reset, the carry
    int p0 = __shfl_up_sync(0xFFFFFFFFu, v0, 1), p1 = __shfl_up_sync(0xFFFFFFFFu, v1, 1), p2 = __shfl_up_sync(0xFFFFFFFFu, v2, 1);
    uint32_t open = !__shfl_up_sync(0xFFFFFFFFu, g, 1);
    if (lane == 0) { p0 = p1 = p2 = 0; open = 1; }
    for (int w = warp - 1; w >= 0 && open; w--) {
        p0 += ws[4 * w]; p1 += ws[4 * w + 1]; p2 += ws[4 * w + 2];
        if (ws[4 * w + 3]) open = 0;
    }
    if (open) { p0 += carry[0]; p1 += carry[1]; p2 += carry[2]; }
    uint32_t m = b0 / bpm, k = b0 - m * bpm;
    for (uint32_t b = b0; b < b1; b++) {
        if (k == 0 && ResetAt(m, ri)) p0 = p1 = p2 = 0;
        const int d = LoadDc(rec + b);
        const uint32_t comp = (comp_bits >> (2 * k)) & 3u;
        p0 += comp == 0u ? d : 0;
        p1 += comp == 1u ? d : 0;
        p2 += comp == 2u ? d : 0;
        rec[b].dc = int16_t(comp == 0u ? p0 : comp == 1u ? p1 : p2);
        if (++k == bpm) { k = 0; m++; }
    }
}

__global__ void __launch_bounds__(kDcTileMcus) dc_sums(K1Args a) {
    PdlEntry();
    __shared__ int red[3];
    const int tid = threadIdx.x;
    const uint32_t tile = blockIdx.x;
    const uint32_t img = UpperIndex(a.img_dctile0, uint32_t(a.nimages), tile);
    const ImageDesc& im = a.images[img];
    const int64_t m0 = int64_t(tile - a.img_dctile0[img]) * kDcTileMcus;
    const int64_t m1 = min(m0 + kDcTileMcus, int64_t(im.total_mcus));
    const int64_t reset = LastReset(m0, m1, im.restart_interval);
    const int64_t m = m0 + tid;
    if (tid < 3) red[tid] = 0;
    __syncthreads();
    McuDc mcu;
    mcu.Load(a.blk_rec + im.blk0 + m * im.bpm, im.bpm, im.comp_bits, m < m1 && m >= reset);
    const int s[3] = {mcu.s0, mcu.s1, mcu.s2};
#pragma unroll
    for (int c = 0; c < 3; c++) {
        int v = s[c];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
        if ((tid & 31) == 0 && v) atomicAdd(&red[c], v);
    }
    __syncthreads();
    if (tid == 0) a.dc_partial[tile] = make_int3(red[0], red[1], red[2]);
}

// One CTA per image: exclusive segmented scan over the image's DC-tile sums (a tile that
// contains a predictor reset cuts the chain; its sums already start at its last reset).
__global__ void __launch_bounds__(kScanThreads) dc_scan(K1Args a) {
    PdlEntry();
    __shared__ int s_v[kScanThreads / 32][3];
    __shared__ uint32_t s_f[kScanThreads / 32];
    const uint32_t img = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const ImageDesc& im = a.images[img];
    const uint32_t t0 = a.img_dctile0[img], t1 = a.img_dctile0[img + 1];
    const int ri = im.restart_interval;
    int c0 = 0, c1 = 0, c2 = 0;   // predictors entering the current chunk
    for (uint32_t base = t0; base < t1; base += kScanThreads) {
        const uint32_t k = base + tid;
        int3 part = make_int3(0, 0, 0);
        uint32_t f = 0;
        if (k < t1) {
            part = a.dc_partial[k];
            const int64_t m0 = int64_t(k - t0) * kDcTileMcus;
            f = LastReset(m0, min(m0 + kDcTileMcus, int64_t(im.total_mcus)), ri) >= 0 ? 1u : 0u;
        }
        int v0 = part.x, v1 = part.y, v2 = part.z;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int p0 = __shfl_up_sync(0xFFFFFFFFu, v0, d);
            const int p1 = __shfl_up_sync(0xFFFFFFFFu, v1, d);
            const int p2 = __shfl_up_sync(0xFFFFFFFFu, v2, d);
            const uint32_t pf = __shfl_up_sync(0xFFFFFFFFu, f, d);
            if (lane >= d) {
                if (!f) { v0 += p0; v1 += p1; v2 += p2; }
                f |= pf;
            }
        }
        __syncthreads();
        if (lane == 31) { s_v[warp][0] = v0; s_v[warp][1] = v1; s_v[warp][2] = v2; s_f[warp] = f; }
        __syncthreads();
        int q0 = 0, q1 = 0, q2 = 0;
        uint32_t qf = 0;
        for (int w = 0; w < warp; w++) {
            if (s_f[w]) { q0 = s_v[w][0]; q1 = s_v[w][1]; q2 = s_v[w][2]; } else { q0 += s_v[w][0]; q1 += s_v[w][1]; q2 += s_v[w][2]; }
            qf |= s_f[w];
        }
        if (!qf) { q0 += c0; q1 += c1; q2 += c2; }
        int x0 = __shfl_up_sync(0xFFFFFFFFu, v0, 1), x1 = __shfl_up_sync(0xFFFFFFFFu, v1, 1), x2 = __shfl_up_sync(0xFFFFFFFFu, v2, 1);
        uint32_t xf = __shfl_up_sync(0xFFFFFFFFu, f, 1);
        if (lane == 0) { x0 = x1 = x2 = 0; xf = 0; }
        if (k < t1) a.dc_carry[k] = xf ? make_int3(x0, x1, x2) : make_int3(x0 + q0, x1 + q1, x2 + q2);
        int w0 = 0, w1 = 0, w2 = 0;
        uint32_t wf = 0;
        for (int w = 0; w < kScanThreads / 32; w++) {
            if (s_f[w]) { w0 = s_v[w][0]; w1 = s_v[w][1]; w2 = s_v[w][2]; } else { w0 += s_v[w][0]; w1 += s_v[w][1]; w2 += s_v[w][2]; }
            wf |= s_f[w];
        }
        if (wf) { c0 = w0; c1 = w1; c2 = w2; } else { c0 += w0; c1 += w1; c2 += w2; }
    }
}

__global__ void __launch_bounds__(kDcTileMcus) dc_apply(K1Args a) {
    PdlEntry();
    __shared__ int wsum[8][3];
    __shared__ int wflag[8];
    __shared__ int carry_s[3];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t tile = blockIdx.x;
    const uint32_t img = UpperIndex(a.img_dctile0, uint32_t(a.nimages), tile);
    const ImageDesc& im = a.images[img];
    const uint32_t tile_first = a.img_dctile0[img];
    const int64_t m0 = int64_t(tile - tile_first) * kDcTileMcus;
    const int64_t m1 = min(m0 + kDcTileMcus, int64_t(im.total_mcus));
    const int ri = im.restart_interval;
    const int64_t m = m0 + tid;
    const bool active = m < m1;
    const bool reset_here = active && ResetAt(uint32_t(m), ri);

    BlockRec* rec = a.blk_rec + im.blk0 + m * im.bpm;
    McuDc mcu;
    mcu.Load(rec, im.bpm, im.comp_bits, active);
    // inclusive segmented scan of the per-MCU sums
    int v0 = mcu.s0, v1 = mcu.s1, v2 = mcu.s2;
    uint32_t f = reset_here ? 1u : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int p0 = __shfl_up_sync(0xFFFFFFFFu, v0, d);
        const int p1 = __shfl_up_sync(0xFFFFFFFFu, v1, d);
        const int p2 = __shfl_up_sync(0xFFFFFFFFu, v2, d);
        const uint32_t pf = __shfl_up_sync(0xFFFFFFFFu, f, d);
        if (lane >= d) {
            if (!f) { v0 += p0; v1 += p1; v2 += p2; }
            f |= pf;
        }
    }
    if (lane == 31) { wsum[warp][0] = v0; wsum[warp][1] = v1; wsum[warp][2] = v2; wflag[warp] = int(f); }
    if (tid == 0) {   // predictors entering the tile, prepared by dc_scan
        const int3 cin = a.dc_carry[tile];
        carry_s[0] = cin.x; carry_s[1] = cin.y; carry_s[2] = cin.z;
    }
    __syncthreads();
    bool open = (f == 0);
    int a0 = 0, a1 = 0, a2 = 0;
    for (int w = warp - 1; w >= 0 && open; w--) {
        a0 += wsum[w][0]; a1 += wsum[w][1]; a2 += wsum[w][2];
        if (wflag[w]) open = false;
    }
    if (open) { a0 += carry_s[0]; a1 += carry_s[1]; a2 += carry_s[2]; }
    // exclusive prefix = predictor values entering this MCU; the absolute DC replaces the difference in the
    // block's record (K2 reads end index and DC together)
    if (!active) return;
    mcu.Store(rec, im.bpm, im.comp_bits, reset_here ? 0 : v0 + a0 - mcu.s0, reset_here ? 0 : v1 + a1 - mcu.s1,
              reset_here ? 0 : v2 + a2 - mcu.s2);
}

// Before the separate kernels redo a batch the fused kernel mis-speculated on: what its write pass reported per picture
// ("ran out of bytes") came from wrong start states.
__global__ void k1_clear_short(K1Args a) {
    const int i = int(blockIdx.x * blockDim.x + threadIdx.x);
    if (i < a.nimages) a.status[i].flags &= ~kDecodeShort;
}

template <int S>
cudaError_t SyncImpl(const K1Args& a, int round, cudaStream_t stream, uint32_t* launches) {
    static_assert(S <= 128, "the packed decoder state holds bit positions below 2048");
    const size_t smem = sizeof(K1Smem<S>) + a.lut_smem_bytes;
    if (smem > 48 * 1024) return cudaErrorInvalidValue;   // 3 table pairs + the full second-level arena fit
    if (round >= 0) return LaunchPdl(launches, k1_sync<S>, dim3(a.total_ctas), dim3(T), smem, stream, a, round, T + 1);
    return LaunchPdl(launches, k1_write<S>, dim3(a.total_ctas), dim3(T), smem, stream, a);
}

}  // namespace

cudaError_t LaunchK1Sync(const K1Args& a, int round, cudaStream_t stream, uint32_t* launches) {
    if (a.total_ctas == 0) return cudaSuccess;
    switch (a.sub_bytes) {
        case 32: return SyncImpl<32>(a, round, stream, launches);
        case 64: return SyncImpl<64>(a, round, stream, launches);
        case 128: return SyncImpl<128>(a, round, stream, launches);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t LaunchK1ClearShort(const K1Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.nimages <= 0) return cudaSuccess;
    k1_clear_short<<<dim3((a.nimages + 255) / 256), dim3(256), 0, stream>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) ++*launches;
    return e;
}

cudaError_t LaunchK1Fused(const K1Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_ctas == 0) return cudaSuccess;
    const int max_iters = T + 1;
    switch (a.sub_bytes) {
        case 32: { const size_t smem = sizeof(K1Smem<32>) + a.lut_smem_bytes; if (smem > 48 * 1024) return cudaErrorInvalidValue;
                   return LaunchPdl(launches, a.inline_destuff ? k1_fused<32, true> : k1_fused<32, false>, dim3(a.total_ctas), dim3(T), smem,
                                    stream, a, max_iters); }
        case 64: { const size_t smem = sizeof(K1Smem<64>) + a.lut_smem_bytes; if (smem > 48 * 1024) return cudaErrorInvalidValue;
                   return LaunchPdl(launches, a.inline_destuff ? k1_fused<64, true> : k1_fused<64, false>, dim3(a.total_ctas), dim3(T), smem,
                                    stream, a, max_iters); }
        case 128: { const size_t smem = sizeof(K1Smem<128>) + a.lut_smem_bytes; if (smem > 48 * 1024) return cudaErrorInvalidValue;
                    return LaunchPdl(launches, a.inline_destuff ? k1_fused<128, true> : k1_fused<128, false>, dim3(a.total_ctas), dim3(T), smem,
                                    stream, a, max_iters); }
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t LaunchK1Write(const K1Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_ctas == 0) return cudaSuccess;
    const cudaError_t e = LaunchPdl(launches, k1_scan, dim3(a.nimages), dim3(kScanThreads), 0, stream, a);
    if (e != cudaSuccess) return e;
    switch (a.sub_bytes) {
        case 32: return SyncImpl<32>(a, -1, stream, launches);
        case 64: return SyncImpl<64>(a, -1, stream, launches);
        case 128: return SyncImpl<128>(a, -1, stream, launches);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t LaunchDcScan(const K1Args& a, cudaStream_t stream, uint32_t* launches) {
    if (a.total_dc_tiles == 0) return cudaSuccess;
    cudaError_t e = LaunchPdl(launches, dc_sums, dim3(a.total_dc_tiles), dim3(kDcTileMcus), 0, stream, a);
    if (e == cudaSuccess) e = LaunchPdl(launches, dc_scan, dim3(a.nimages), dim3(kScanThreads), 0, stream, a);
    if (e == cudaSuccess) e = LaunchPdl(launches, dc_apply, dim3(a.total_dc_tiles), dim3(kDcTileMcus), 0, stream, a);
    return e;
}

// Forces the module holding this stage's kernels onto the device (CUDA loads lazily: the first launch
// of every kernel would otherwise pay for it inside the first decode call).
cudaError_t PreloadK1() {
    cudaFuncAttributes at;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_sync<128>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_sync<64>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_sync<32>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_write<128>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_write<64>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_write<32>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<128, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<128, true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<64, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<64, true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<32, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_fused<32, true>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, k1_scan);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, dc_sums);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, dc_scan);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&at, dc_apply);
    return e;
}

}  // namespace rjb
