// jpeg_parser.cpp — see jpeg_parser.h. Accept/reject rules follow
// src/rocjpeg_parser.cpp of the reference (line numbers cited inline).
#include "jpeg_parser.h"
#include "huff_core.cuh"

#include <cuda_runtime_api.h>

#include <atomic>
#include <memory>
#include <mutex>
#include <vector>

#include <string>

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>

namespace rjb {

namespace {
constexpr int kStatusSuccess = 0;
constexpr int kStatusBadJpeg = -3;
constexpr int kStatusNotSupported = -4;

const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                             41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                             30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

inline uint32_t Rd16(const uint8_t* p) { return (uint32_t(p[0]) << 8) | p[1]; }
inline size_t Align16(size_t v) { return (v + 15) & ~size_t(15); }
}  // namespace

int PoisonByte() {
    const char* v = std::getenv("ROCJPEG_B200_POISON");
    return (v && *v) ? int(std::strtol(v, nullptr, 0) & 0xFF) : -1;
}

// ------------------------------------------------------------ StagingBuffer

StagingBuffer::~StagingBuffer() { Release(); }

void StagingBuffer::Release() {
    if (!ptr_) return;
    if (pinned_) {
        cudaFreeHost(ptr_);
    } else {
        std::free(ptr_);
    }
    ptr_ = nullptr;
    cap_ = 0;
    pinned_ = false;
}

uint8_t* StagingBuffer::Reserve(size_t bytes) {
    if (bytes <= cap_) return ptr_;
    Release();
    size_t want = (bytes + bytes / 4 + 4095) & ~size_t(4095);
    void* p = nullptr;
    // Page-locked + portable so any device's stream can DMA from it, mapped so a
    // gather kernel can read it in place. Falls back to pageable memory when no
    // CUDA driver is present (host-only unit tests); decode still works from it.
    cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable | cudaHostAllocMapped);
    if (e == cudaSuccess && p) {
        pinned_ = true;
    } else {
        (void)cudaGetLastError();
        p = nullptr;
        if (posix_memalign(&p, 4096, want) != 0) p = nullptr;
        pinned_ = false;
    }
    if (!p) {
        cap_ = 0;
        return nullptr;
    }
    ptr_ = static_cast<uint8_t*>(p);
    cap_ = want;
    if (const int poison = PoisonByte(); poison >= 0) std::memset(ptr_, poison, cap_);
    return ptr_;
}

// ------------------------------------------------------------ PinnedPool

namespace {
constexpr size_t kMinBlockLog2 = 12;               // 4 KiB
constexpr size_t kFirstSlab = size_t(16) << 20;    // doubles up to kMaxSlab
constexpr size_t kMaxSlab = size_t(256) << 20;
inline int Log2Ceil(size_t v) {
    int l = 0;
    while ((size_t(1) << l) < v) l++;
    return l;
}

inline uint8_t* Poisoned(void* p, size_t bytes) {   // a block recycled from the free list too (ROCJPEG_B200_POISON)
    if (const int poison = PoisonByte(); p && poison >= 0) std::memset(p, poison, bytes);
    return static_cast<uint8_t*>(p);
}
}  // namespace

PinnedPool& PinnedPool::Get() {
    static PinnedPool* pool = new PinnedPool();   // never destroyed: handles may outlive static destructors
    return *pool;
}

uint8_t* PinnedPool::Alloc(size_t bytes, size_t* cap, bool* pinned) {
    const int cls = std::max<int>(Log2Ceil(bytes ? bytes : 1), int(kMinBlockLog2));
    const size_t want = size_t(1) << cls;
    std::lock_guard<std::mutex> lock(m_);
    if (free_.size() <= size_t(cls)) free_.resize(size_t(cls) + 1);
    *cap = want;
    if (!free_[size_t(cls)].empty()) {
        uint8_t* p = free_[size_t(cls)].back();
        free_[size_t(cls)].pop_back();
        *pinned = true;
        return Poisoned(p, want);
    }
    if (!no_driver_ && slab_left_ < want) {
        // the tail of the old slab is abandoned (at most half of it, the slabs double)
        if (next_slab_ == 0) {
            const char* mb = std::getenv("ROCJPEG_B200_PINNED_SLAB_MB");
            next_slab_ = (mb && *mb) ? std::max<size_t>(1, size_t(std::atoi(mb))) << 20 : kFirstSlab;
        }
        const size_t slab = std::max(next_slab_, want);
        void* p = nullptr;
        cudaError_t e = cudaHostAlloc(&p, slab, cudaHostAllocPortable | cudaHostAllocMapped);
        if (e == cudaSuccess && p) {
            slab_ = static_cast<uint8_t*>(p);
            slab_left_ = slab;
            next_slab_ = std::min(kMaxSlab, slab * 2);
        } else {
            (void)cudaGetLastError();
            if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorNotSupported) no_driver_ = true;
            slab_left_ = 0;
        }
    }
    if (slab_left_ >= want) {
        uint8_t* p = slab_;
        slab_ += want;
        slab_left_ -= want;
        *pinned = true;
        return Poisoned(p, want);
    }
    // no CUDA driver (host-only unit tests) or page-locking failed: pageable memory, decode still works from it
    void* p = nullptr;
    if (posix_memalign(&p, 4096, want) != 0) p = nullptr;
    *pinned = false;
    return Poisoned(p, want);
}

void PinnedPool::Free(uint8_t* p, size_t cap, bool pinned) {
    if (!p) return;
    if (!pinned) {
        std::free(p);
        return;
    }
    const int cls = Log2Ceil(cap);
    std::lock_guard<std::mutex> lock(m_);
    if (free_.size() <= size_t(cls)) free_.resize(size_t(cls) + 1);
    free_[size_t(cls)].push_back(p);
}

void PooledBuffer::Release() {
    if (ptr_) PinnedPool::Get().Free(ptr_, cap_, pinned_);
    ptr_ = nullptr;
    cap_ = 0;
    pinned_ = false;
}

uint8_t* PooledBuffer::Reserve(size_t bytes) {
    if (bytes <= cap_ && ptr_) return ptr_;
    Release();
    ptr_ = PinnedPool::Get().Alloc(bytes, &cap_, &pinned_);
    if (!ptr_) cap_ = 0;
    return ptr_;
}

// ------------------------------------------------------------ classification

// src/rocjpeg_parser.cpp:432-470
int ClassifyChromaSubsampling(const int32_t h[3], const int32_t v[3]) {
    auto is = [&](int h0, int h1, int h2, int v0, int v1, int v2) {
        return h[0] == h0 && h[1] == h1 && h[2] == h2 && v[0] == v0 && v[1] == v1 && v[2] == v2;
    };
    if (is(1, 1, 1, 1, 1, 1) || is(2, 2, 2, 2, 2, 2) || is(4, 4, 4, 4, 4, 4)) return CSS_444;
    if (is(1, 1, 1, 2, 1, 1)) return CSS_440;
    if (is(2, 1, 1, 1, 1, 1) || is(2, 1, 1, 2, 2, 2) || is(2, 2, 2, 2, 1, 1)) return CSS_422;
    if (is(2, 1, 1, 2, 1, 1)) return CSS_420;
    if (is(4, 1, 1, 1, 1, 1)) return CSS_411;
    if (is(1, 0, 0, 1, 0, 0) || is(4, 0, 0, 4, 0, 0)) return CSS_400;
    return CSS_UNKNOWN;
}

// ------------------------------------------------------------ Huffman tables

// T.81 Annex C (code assignment) + F.2.2.3 (decoder tables), restated as a two-level lookup over
// a left-aligned peek (device_types.h: HuffLutSet). slot: t = DC table t, kHuffIds + t = AC table t.
// Sub-tables are appended to out->sub (the caller zeroes the set before building its tables).
void BuildHuffLut(const HuffSpec& spec, int slot, HuffLutSet* out, uint32_t sub_cap) {
    uint32_t* fast = out->fast[slot];
    if (sub_cap > uint32_t(kSubCap)) sub_cap = uint32_t(kSubCap);
    const bool is_ac = slot >= kHuffIds;
    const uint32_t invalid = MakeEntry(16, 0, is_ac);   // unassigned code: 16 bits consumed, symbol 0
    for (int i = 0; i < kFastSize; i++) fast[i] = invalid;
    std::memcpy(out->vals[slot], spec.vals, 256);
    struct Long { uint32_t code, len, sym; };
    std::vector<Long> longs;
    uint32_t code = 0, k = 0;
    for (int l = 1; l <= 16; l++) {
        out->valoff[slot][l] = int32_t(k) - int32_t(code);
        for (uint32_t i = 0; i < spec.bits[l - 1]; i++, code++, k++) {
            if (code >= (1u << l) || k >= 256) continue;   // over-subscribed DHT: the excess codes cannot occur
            if (l <= kFastBits) {
                const uint32_t first = code << (kFastBits - l);
                const uint32_t entry = MakeEntry(uint32_t(l), spec.vals[k], is_ac);
                for (uint32_t j = 0; j < (1u << (kFastBits - l)); j++) fast[first + j] = entry;
            } else {
                longs.push_back(Long{code, uint32_t(l), spec.vals[k]});
            }
        }
        uint32_t up = code << (16 - l);
        out->upper[slot][l] = up > 0x10000u ? 0x10000u : up;
        code <<= 1;
    }
    out->upper[slot][0] = 0;
    out->valoff[slot][0] = 0;
    // second level: one sub-table per first-level prefix that has longer codes under it, indexed by
    // the next (longest code under the prefix - kFastBits) bits. Canonical codes are assigned in
    // increasing order, so the codes of one prefix are contiguous in `longs`.
    for (size_t i = 0; i < longs.size();) {
        const uint32_t prefix = longs[i].code >> (longs[i].len - kFastBits);
        size_t j = i;
        uint32_t maxlen = 0;
        while (j < longs.size() && (longs[j].code >> (longs[j].len - kFastBits)) == prefix) maxlen = std::max(maxlen, longs[j++].len);
        const uint32_t x = maxlen - kFastBits, n = 1u << x;
        if (out->sub_used + n > sub_cap) {
            fast[prefix] = MakeLink(0, 0);   // arena exhausted: the canonical search resolves these codes
        } else {
            const uint32_t first = out->sub_used;
            out->sub_used += n;
            for (uint32_t t = 0; t < n; t++) out->sub[first + t] = invalid;
            for (size_t q = i; q < j; q++) {
                const uint32_t rest = longs[q].len - kFastBits;   // bits of the code below the prefix
                const uint32_t low = (longs[q].code & ((1u << rest) - 1u)) << (x - rest);
                const uint32_t entry = MakeEntry(longs[q].len, longs[q].sym, is_ac);
                for (uint32_t t = 0; t < (1u << (x - rest)); t++) out->sub[first + low + t] = entry;
            }
            fast[prefix] = MakeLink(x, first);
        }
        i = j;
    }
}

// ------------------------------------------------------------ StreamParser

bool StreamParser::TablesFailed() {
    dht_cache_.key.clear();
    dqt_cache_.key.clear();
    lut_valid_ = false;
    p_.valid = false;
    return false;
}

bool StreamParser::Fail(const char* why) {
    err_ = why;
    p_.valid = false;
    return false;
}

// src/rocjpeg_parser.cpp:160-207
bool StreamParser::ParseSof(const uint8_t* s, uint32_t seglen, bool extended) {
    if (seglen < 8) return Fail("truncated SOF");
    if (extended) {   // SOF1: the sequential Huffman process; the same decode as SOF0 when the samples have 8 bits
        if (s[2] != 8) return Fail("not a baseline JPEG: extended sequential frame (SOF1) with 12-bit samples - only 8-bit samples are decoded");
        p_.features |= kFeatSof1;
    }
    p_.height = int32_t(Rd16(s + 3));
    p_.width = int32_t(Rd16(s + 5));
    p_.ncomp = s[7];
    if (p_.ncomp > 3) return Fail("more than three components");                // :172
    if (seglen < 8u + 3u * uint32_t(p_.ncomp)) return Fail("truncated SOF");
    for (int i = 0; i < p_.ncomp; i++) {
        p_.comp_id[i] = s[8 + 3 * i];
        uint8_t sf = s[9 + 3 * i], tq = s[10 + 3 * i];
        if (tq >= 4) return Fail("quantiser table selector out of range");     // :185
        p_.hs[i] = sf >> 4;
        p_.vs[i] = sf & 15;
        p_.tq[i] = tq;
    }
    int h0 = p_.hs[0] ? p_.hs[0] : 1, v0 = p_.vs[0] ? p_.vs[0] : 1;
    p_.num_mcus_ref = uint32_t((p_.width + h0 * 8 - 1) / (h0 * 8)) * uint32_t((p_.height + v0 * 8 - 1) / (v0 * 8));  // :197
    p_.css = ClassifyChromaSubsampling(p_.hs, p_.vs);
    return true;
}

// src/rocjpeg_parser.cpp:256-313
bool StreamParser::ParseDht(const uint8_t* payload, uint32_t n) {
    int32_t rem = int32_t(n);
    const uint8_t* q = payload;
    while (rem > 0) {
        if (rem < 17) return Fail("truncated DHT");
        uint8_t idx = *q++;
        bool is_ac = (idx & 0xF0) != 0;
        int id = idx & 0x0F;
        if (id >= kHuffIds) return Fail("Huffman table id out of range");     // T.81 B.2.4.2: Th 0..3 (the reference stops at 1, :274)
        if (id >= 2) p_.features |= kFeatHuffId23;
        uint32_t count = 0;
        for (int i = 0; i < 16; i++) count += q[i];
        if (is_ac ? count > 162 : count > 12) return Fail("too many Huffman values");   // :291, :298
        if (int32_t(17 + count) > rem) return Fail("truncated DHT");
        HuffSpec& t = is_ac ? p_.ac[id] : p_.dc[id];
        std::memset(&t, 0, sizeof(t));
        std::memcpy(t.bits, q, 16);
        std::memcpy(t.vals, q + 16, count);
        t.count = count;
        t.present = true;
        q += 16 + count;
        rem -= 17 + int32_t(count);
    }
    return true;
}

// src/rocjpeg_parser.cpp:217-246
bool StreamParser::ParseDqt(const uint8_t* payload, uint32_t n) {
    const uint8_t *q = payload, *end = payload + n;
    while (q < end) {
        uint8_t idx = *q++;
        const int wide = idx >> 4;   // Pq: 0 = 8-bit steps, 1 = 16-bit (the reference rejects those, :230)
        idx &= 15;
        if (wide > 1) return Fail("quantisation table precision out of range");
        if (idx >= 4) return Fail("quantisation table id out of range");             // :234
        if (q + (wide ? 128 : 64) > end) return Fail("truncated DQT");
        for (int k = 0; k < 64; k++) p_.qt[idx][k] = wide ? uint16_t(Rd16(q + 2 * k)) : uint16_t(q[k]);
        if (wide) p_.features |= kFeatDqt16;
        p_.qt_present[idx] = true;
        q += wide ? 128 : 64;
    }
    return true;
}

// One DHT / DQT segment of the stream being parsed. While it repeats the previous stream's bytes nothing happens;
// at the first difference the tables are cleared and every segment seen so far is parsed for real.
template <class ParseFn, class ClearFn>
bool StreamParser::TakeTableSegment(TableCache& c, const uint8_t* payload, uint32_t n, ParseFn parse, ClearFn clear) {
    if (c.nseg < 8) {
        c.seg[c.nseg] = payload;
        c.seglen[c.nseg] = n;
    }
    c.nseg++;
    if (c.matching) {
        if (c.nseg <= 8 && c.cursor + n <= c.key.size() && std::memcmp(c.key.data() + c.cursor, payload, n) == 0) {
            c.cursor += n;
            return true;
        }
        c.matching = false;   // diverged: what matched so far belongs to tables that no longer apply
        c.changed = true;
        c.key.clear();
        clear();
        for (int i = 0; i + 1 < c.nseg && i < 8; i++)
            if (!parse(c.seg[i], c.seglen[i])) return false;
    } else if (!c.changed) {
        c.changed = true;
        c.key.clear();
        clear();
    }
    return parse(payload, n);
}

// All table segments of the stream have been seen: a stream that only repeated a prefix of the previous one's
// is re-parsed; the key of the next comparison is this stream's.
template <class ParseFn, class ClearFn>
bool StreamParser::FinishTableSegments(TableCache& c, ParseFn parse, ClearFn clear) {
    if (c.matching && c.cursor == c.key.size()) return true;   // identical tables: everything derived from them stands
    if (c.matching) {
        c.matching = false;
        c.changed = true;
        clear();
        for (int i = 0; i < c.nseg && i < 8; i++)
            if (!parse(c.seg[i], c.seglen[i])) {
                c.key.clear();
                return false;
            }
    }
    c.key.clear();
    if (c.nseg <= 8)
        for (int i = 0; i < c.nseg; i++) c.key.insert(c.key.end(), c.seg[i], c.seg[i] + c.seglen[i]);
    return true;
}

// src/rocjpeg_parser.cpp:324-363
bool StreamParser::ParseSos(const uint8_t* s, uint32_t seglen) {
    if (seglen < 3) return Fail("truncated SOS");
    int n = s[2];
    if (n > 3) return Fail("more than three scan components");                     // :333
    if (seglen < 6u + 2u * uint32_t(n)) return Fail("truncated SOS");
    p_.scan_ncomp = n;
    for (int i = 0; i < n; i++) {
        uint8_t cid = s[3 + 2 * i], t = s[4 + 2 * i];
        if ((t & 15) >= 4 || (t >> 4) >= 4) return Fail("Huffman selector out of range");   // :347-354
        if (cid != p_.comp_id[i]) return Fail("scan components do not follow the frame order");  // :355
        p_.td[i] = t >> 4;
        p_.ta[i] = t & 15;
    }
    return true;
}

void StreamParser::DeriveGeometry() {
    p_.hmax = p_.vmax = 1;
    p_.mcus_x = p_.mcus_y = p_.bpm = 0;
    for (int i = 0; i < 3; i++) p_.blocks_w[i] = p_.blocks_h[i] = 0;
    if (p_.ncomp < 1 || p_.width <= 0 || p_.height <= 0) return;
    for (int i = 0; i < p_.ncomp; i++) {
        if (p_.hs[i] > p_.hmax) p_.hmax = p_.hs[i];
        if (p_.vs[i] > p_.vmax) p_.vmax = p_.vs[i];
    }
    if (p_.ncomp == 1) {
        // single-component scan: MCU = one 8x8 block, sampling factors ignored (T.81 A.2.2)
        p_.mcus_x = (p_.width + 7) / 8;
        p_.mcus_y = (p_.height + 7) / 8;
        p_.bpm = 1;
        p_.blocks_w[0] = p_.mcus_x;
        p_.blocks_h[0] = p_.mcus_y;
    } else {
        p_.mcus_x = (p_.width + 8 * p_.hmax - 1) / (8 * p_.hmax);
        p_.mcus_y = (p_.height + 8 * p_.vmax - 1) / (8 * p_.vmax);
        for (int i = 0; i < p_.ncomp; i++) {
            p_.blocks_w[i] = p_.mcus_x * p_.hs[i];
            p_.blocks_h[i] = p_.mcus_y * p_.vs[i];
            p_.bpm += p_.hs[i] * p_.vs[i];
        }
    }
}

// Host restatement of the GPU destuffing pass (k0_destuff.cu) over the entropy-coded bytes `d[0, length)`:
// finds the first FF D9 (the reference's ParseEOI, parser.cpp:400-416) and writes the destuffed,
// marker-free bitstream, one 16-byte-aligned segment per restart interval. Rules (T.81 B.1.1.5, E.1.4;
// the tolerant ones are this decoder's, shared with the GPU pass):
//   FF 00 -> data byte FF;  FF FF -> the first FF is a fill byte;  FF D0..D7 -> ends the interval;
//   FF D9 -> ends the slice;  FF xx (any other marker) -> the rest of the interval carries no data;
//   a lone FF at the very end carries no data; intervals beyond ParsedJpeg::nseg are dropped, missing
//   ones are empty.
void StreamParser::ExtractEntropyData(const uint8_t* d, size_t length, HostScan* hs) const {
    hs->segments.clear();
    hs->restart_markers_seen = 0;
    const size_t expected = p_.nseg;
    const size_t cap = length + (expected + 2) * 48 + 64;
    hs->clean.assign(cap, 0);
    uint8_t* out = hs->clean.data();
    size_t o = 0, seg_start = 0, pos = 0;
    bool dead = false;   // a non-restart marker was met: no more data until the next RSTn
    auto close_segment = [&]() {
        if (hs->segments.size() < expected) hs->segments.push_back(Segment{uint32_t(seg_start), uint32_t(o - seg_start)});
        size_t padded = Align16(o) + 16;   // zero tail: the bit reader may look 16 bytes ahead
        std::memset(out + o, 0, padded - o);
        o = padded;
        seg_start = o;
    };
    size_t eoi = length;
    while (pos < length) {
        const uint8_t* q = static_cast<const uint8_t*>(std::memchr(d + pos, 0xFF, length - pos));
        size_t stop = q ? size_t(q - d) : length;
        if (!dead && stop > pos && o + (stop - pos) + 64 <= cap) {
            std::memcpy(out + o, d + pos, stop - pos);
            o += stop - pos;
        }
        pos = stop;
        if (!q) break;
        if (pos + 1 >= length) {   // lone FF at the very end: belongs to the slice, carries no data
            pos = length;
            break;
        }
        uint8_t nx = d[pos + 1];
        if (nx == 0x00) {
            if (!dead && o + 65 <= cap) out[o++] = 0xFF;
            pos += 2;
        } else if (nx == 0xD9) {
            eoi = pos;
            break;
        } else if ((nx & 0xF8) == 0xD0) {
            hs->restart_markers_seen++;
            if (o + 48 + 64 <= cap) close_segment();
            dead = false;
            pos += 2;
        } else if (nx == 0xFF) {
            pos += 1;   // fill byte
        } else {
            dead = true;   // any other marker ends the entropy-coded data of this interval
            pos += 2;
        }
    }
    hs->scan_size = uint32_t(eoi);   // no EOI: the slice runs to the end of the buffer
    close_segment();
    while (hs->segments.size() < expected && o + 48 + 64 <= cap) close_segment();   // missing intervals: empty
    hs->clean_bytes = o;
    hs->done = true;
}

const HostScan& StreamParser::host_scan() const {
    std::lock_guard<std::mutex> lock(mutex_);
    EnsureStagedLocked();
    if (!host_scan_.done && p_.valid && raw_.host) ExtractEntropyData(raw_.host, raw_.nbytes, &host_scan_);
    return host_scan_;
}

namespace {
// cuPointerGetAttributes of the driver, reached through the runtime (no link dependency on libcuda): one call
// answers "page-locked? device alias? which allocation?" and does not fail on ordinary host pointers.
typedef int (*PointerAttributesFn)(unsigned int, int*, void**, unsigned long long);
PointerAttributesFn DriverPointerAttributes() {
    static const PointerAttributesFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuPointerGetAttributes", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            (void)cudaGetLastError();
            f = nullptr;
        }
        return reinterpret_cast<PointerAttributesFn>(f);
    }();
    return fn;
}

// Is `p` page-locked host memory the device can read in place? Returns its device alias or nullptr, and the
// allocation it belongs to.
const uint8_t* DeviceAliasOf(const uint8_t* p, uintptr_t* range_base, size_t* range_size) {
    static std::atomic<int> no_driver{0};
    static const bool enabled = [] {
        const char* v = std::getenv("ROCJPEG_B200_ZERO_COPY");
        return !(v && *v == '0');
    }();
    *range_base = 0;
    *range_size = 0;
    if (!enabled || no_driver.load(std::memory_order_relaxed)) return nullptr;
    if (PointerAttributesFn fn = DriverPointerAttributes()) {
        // CU_POINTER_ATTRIBUTE_MEMORY_TYPE = 2, DEVICE_POINTER = 3, RANGE_START_ADDR = 11, RANGE_SIZE = 12, IS_MANAGED = 8
        int which[5] = {2, 3, 11, 12, 8};
        unsigned int mem_type = 0;
        unsigned long long dev_ptr = 0, start = 0;
        size_t size = 0;
        unsigned int managed = 0;
        void* out[5] = {&mem_type, &dev_ptr, &start, &size, &managed};
        if (fn(5, which, out, static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(p))) == 0) {
            if (mem_type == 1u /* CU_MEMORYTYPE_HOST */ && dev_ptr != 0 && !managed) {
                const uintptr_t a = reinterpret_cast<uintptr_t>(p);
                if (start != 0 && size != 0 && a >= uintptr_t(start) && a < uintptr_t(start) + size) {
                    *range_base = uintptr_t(start);
                    *range_size = size;
                }
                return reinterpret_cast<const uint8_t*>(uintptr_t(dev_ptr));
            }
            if (mem_type == 0u) return nullptr;   // an ordinary host pointer
        }
        // anything else (driver not initialised yet, managed memory ...): ask the runtime, which initialises itself
    }
    cudaPointerAttributes at;
    cudaError_t e = cudaPointerGetAttributes(&at, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorNotSupported) no_driver.store(1, std::memory_order_relaxed);
        return nullptr;
    }
    if (at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged) return static_cast<const uint8_t*>(at.devicePointer);
    return nullptr;
}
}  // namespace

// Makes the entropy-coded bytes reachable by the device: in place when the caller's buffer is page-locked,
// otherwise through one copy into pooled page-locked staging (the only per-byte work of a parse).
void StreamParser::AdoptSource(const uint8_t* scan, size_t nbytes) {
    raw_ = RawScan();
    pending_src_ = nullptr;
    pending_len_ = 0;
    raw_.nbytes = uint32_t(nbytes);
    if (const uint8_t* dev = DeviceAliasOf(scan, &raw_.range_base, &raw_.range_size)) {
        raw_.host = scan;
        raw_.dev = dev;
        raw_.zero_copy = true;
        return;
    }
    uint8_t* st = staging_.Reserve(nbytes + 64);
    if (!st) return;   // raw_.host stays null: the decode reports OUT_OF_MEMORY
    std::memset(st + nbytes, 0xFF, 64 - (nbytes & 15));   // what the upload rounds up to
    raw_.host = st;
    raw_.dev = staging_.pinned() ? st : nullptr;
    if (raw_.dev) (void)DeviceAliasOf(st, &raw_.range_base, &raw_.range_size);   // the pool's slab
    // The copy: here, on the caller's thread (default: callers that want it parallel parse from several threads, one handle
    // each, as the reference's perf sample does) - or, with ROCJPEG_B200_DEFERRED_COPY=1, inside the decode call, by its helper
    // threads, chunk by chunk ahead of each chunk's upload (a single-threaded caller with a large pageable batch: c3 1.9 -> 1.1 ms
    // per batch, c4 26.6 -> 7.2 ms; but helper threads of several handles decoding at once oversubscribe a small host, and the
    // caller's buffer must then stay valid until the decode returns, which is all the reference promises anyway).
    const char* dv = std::getenv("ROCJPEG_B200_DEFERRED_COPY");
    pending_src_ = scan;
    pending_len_ = nbytes;
    if (!(dv && *dv == '1') || !raw_.dev) EnsureStagedLocked();
}

void StreamParser::EnsureStagedLocked() const {
    if (!pending_src_) return;
    std::memcpy(const_cast<uint8_t*>(raw_.host), pending_src_, pending_len_);
    pending_src_ = nullptr;
    pending_len_ = 0;
}

void StreamParser::EnsureStaged() const {
    std::lock_guard<std::mutex> lock(mutex_);   // (the same handle may sit in a batch twice: two helper threads)
    EnsureStagedLocked();
}

void StreamParser::BuildDecodeTables() {
    // support check: what the CUDA path decodes (baseline, one interleaved scan
    // over all components, css in {444, 440, 422, 420, 411, 400})
    p_.support_status = kStatusSuccess;
    if (p_.width <= 0 || p_.height <= 0) p_.support_status = kStatusNotSupported;
    else if (p_.ncomp != 1 && p_.ncomp != 3) p_.support_status = kStatusNotSupported;
    else if (p_.scan_ncomp != p_.ncomp) p_.support_status = kStatusNotSupported;
    else if (p_.css == CSS_UNKNOWN) p_.support_status = kStatusNotSupported;
    else if (p_.bpm > kMaxBlocksPerMcu || p_.bpm < 1) p_.support_status = kStatusNotSupported;
    else if (p_.css == CSS_422 && p_.ncomp == 3 && p_.hs[1] == p_.hs[0]) p_.support_status = kStatusNotSupported;
    // A block takes at least two bits (a DC code and an end-of-block): a frame header that announces far more
    // blocks than the bytes present could ever hold (a 100-byte file "of" 65535 x 65535 samples) is not a
    // truncated picture but a bad one - nothing is sized from such a header.
    else if (uint64_t(p_.mcus_x) * uint64_t(p_.mcus_y) * uint64_t(p_.bpm) > 256ull * uint64_t(p_.raw_bytes) + 65536ull)
        p_.support_status = kStatusBadJpeg;
    if (p_.support_status == kStatusSuccess) {
        for (int i = 0; i < p_.ncomp; i++) {
            if (!p_.qt_present[p_.tq[i]]) p_.support_status = kStatusBadJpeg;
            if (!p_.dc[p_.td[i]].present || !p_.ac[p_.ta[i]].present) p_.support_status = kStatusBadJpeg;
        }
    }
    if (dqt_cache_.changed)
        for (int t = 0; t < 4; t++)
            for (int k = 0; k < 64; k++) p_.qt_natural[t][kZigzag[k]] = p_.qt[t][k];
    if (!dht_cache_.changed && lut_valid_) return;   // same DHT bytes as the previous stream: hash, bounds and LUTs stand
    // Identity of the four Huffman tables (batch de-duplication in the decoder).
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](const void* ptr, size_t n) {
        const uint8_t* b = static_cast<const uint8_t*>(ptr);
        for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
    };
    for (int t = 0; t < kHuffIds; t++) {
        uint8_t present[2] = {uint8_t(p_.dc[t].present), uint8_t(p_.ac[t].present)};
        mix(present, 2);
        mix(p_.dc[t].bits, 16);
        mix(p_.dc[t].vals, p_.dc[t].count);
        mix(p_.ac[t].bits, 16);
        mix(p_.ac[t].vals, p_.ac[t].count);
    }
    p_.lut_hash = h;
    // Shortest symbol that carries magnitude bits: code length + SSSS. Bounds how many
    // coefficient entries a scan of a given size can produce.
    uint32_t min_bits = 32;
    for (int t = 0; t < kHuffIds; t++)
        for (int is_ac = 0; is_ac < 2; is_ac++) {
            const HuffSpec& sp = is_ac ? p_.ac[t] : p_.dc[t];
            if (!sp.present) continue;
            uint32_t k = 0;
            for (uint32_t l = 1; l <= 16; l++)
                for (uint32_t i = 0; i < sp.bits[l - 1] && k < 256; i++, k++) {
                    const uint32_t sz = sp.vals[k] & 15u;
                    if (sz && l + sz < min_bits) min_bits = l + sz;
                }
        }
    p_.min_entry_bits = min_bits < 2 ? 2 : (min_bits > 31 ? 2 : min_bits);
    // debug knob: a smaller second-level arena forces long codes onto the canonical search
    const char* cap_env = std::getenv("ROCJPEG_B200_SUBCAP");
    const uint32_t cap = (cap_env && *cap_env) ? uint32_t(std::atoi(cap_env)) : uint32_t(kSubCap);
    // Decoder-form tables are a pure function of the DHT content: a process-wide cache lets every handle that meets the
    // same tables share ONE copy (the reference's perf sample creates one handle per image; 256 first parses took 4.2 ms,
    // most of it building the tables and faulting in the 22 KiB each handle used to keep of its own).
    struct Cached {
        uint64_t hash;
        uint32_t cap;
        HuffSpec dc[kHuffIds], ac[kHuffIds];
        std::shared_ptr<const HuffLutSet> lut;
    };
    static std::mutex cache_mutex;
    static std::vector<std::unique_ptr<Cached>> cache;
    {
        std::lock_guard<std::mutex> lock(cache_mutex);
        for (const auto& c : cache)
            if (c->hash == h && c->cap == cap && std::memcmp(c->dc, p_.dc, sizeof(p_.dc)) == 0 && std::memcmp(c->ac, p_.ac, sizeof(p_.ac)) == 0) {
                lut_ = c->lut;
                lut_cap_ = cap;
                lut_valid_ = true;
                return;
            }
    }
    std::shared_ptr<HuffLutSet> built(new HuffLutSet());
    std::memset(built.get(), 0, sizeof(HuffLutSet));
    for (int t = 0; t < kHuffIds; t++) {
        if (p_.dc[t].present) BuildHuffLut(p_.dc[t], t, built.get(), cap);
        if (p_.ac[t].present) BuildHuffLut(p_.ac[t], kHuffIds + t, built.get(), cap);
    }
    lut_ = built;
    lut_cap_ = cap;
    lut_valid_ = true;
    {
        std::unique_ptr<Cached> c(new Cached);
        c->hash = h;
        c->cap = cap;
        std::memcpy(c->dc, p_.dc, sizeof(p_.dc));
        std::memcpy(c->ac, p_.ac, sizeof(p_.ac));
        c->lut = lut_;
        std::lock_guard<std::mutex> lock(cache_mutex);
        if (cache.size() >= 16) cache.erase(cache.begin());   // oldest out (handles that use it keep their reference)
        cache.push_back(std::move(c));
    }
}

const HuffLutSet& StreamParser::EmptyLut() {
    static const HuffLutSet* empty = [] {
        HuffLutSet* e = new HuffLutSet();
        std::memset(e, 0, sizeof(HuffLutSet));
        return e;
    }();
    return *empty;
}

// Everything of the previous stream except its tables (the reference zeroes its parameters on every parse,
// parser.cpp:54; the tables are compared segment by segment instead, see TableCache).
void StreamParser::ResetFrame() {
    p_.valid = false;
    p_.width = p_.height = p_.ncomp = 0;
    p_.css = CSS_UNKNOWN;
    for (int i = 0; i < 3; i++) p_.comp_id[i] = p_.hs[i] = p_.vs[i] = p_.tq[i] = p_.td[i] = p_.ta[i] = p_.blocks_w[i] = p_.blocks_h[i] = 0;
    p_.scan_ncomp = p_.restart_interval = 0;
    p_.num_mcus_ref = p_.scan_offset = p_.raw_bytes = 0;
    p_.hmax = p_.vmax = 1;
    p_.mcus_x = p_.mcus_y = p_.bpm = 0;
    p_.support_status = 0;
    p_.nseg = 1;
    p_.features &= (kFeatDqt16 | kFeatHuffId23);   // what the kept tables use stays with them; the frame's part is per stream
    raw_ = RawScan();
    pending_src_ = nullptr;
    pending_len_ = 0;
    host_scan_.done = false;
    err_.clear();
    dht_cache_.Begin();
    dqt_cache_.Begin();
}

bool StreamParser::Parse(const uint8_t* d, size_t len) {
    std::lock_guard<std::mutex> lock(mutex_);
    return ParseLocked(d, len, false);
}

int StreamParser::ParseFile(const char* path) {
    std::lock_guard<std::mutex> lock(mutex_);
    ResetFrame();
    FILE* f = path ? std::fopen(path, "rb") : nullptr;
    if (!f) {
        Fail("cannot open the file");
        return -2;
    }
    std::fseek(f, 0, SEEK_END);
    const long size = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    uint8_t* buf = size > 0 ? file_.Reserve(size_t(size) + 64) : nullptr;
    const size_t got = buf ? std::fread(buf, 1, size_t(size), f) : 0;
    std::fclose(f);
    if (!buf || got != size_t(size)) {
        Fail(size <= 0 ? "empty file" : "cannot read the file");
        return -2;
    }
    std::memset(buf + size, 0xFF, 64 - (size_t(size) & 15));   // what the upload rounds up to
    return ParseLocked(buf, size_t(size), true) ? 0 : -3;
}

bool StreamParser::ParseLocked(const uint8_t* d, size_t len, bool data_is_file_buffer) {
    ResetFrame();
    if (!d || len < 4) return Fail("stream too short");
    if (d[0] != 0xFF || d[1] != 0xD8) return Fail("missing SOI");                   // parser.cpp:64
    size_t p = 2;
    bool seen_dht = false, seen_dqt = false, seen_sos = false, seen_sof0 = false;
    auto parse_dht = [this](const uint8_t* q, uint32_t n) { return ParseDht(q, n); };
    auto parse_dqt = [this](const uint8_t* q, uint32_t n) { return ParseDqt(q, n); };
    auto clear_dht = [this]() {
        for (int t = 0; t < kHuffIds; t++) p_.dc[t].present = p_.ac[t].present = false;
        lut_valid_ = false;
        p_.features &= ~kFeatHuffId23;
    };
    auto clear_dqt = [this]() {
        for (int t = 0; t < 4; t++) p_.qt_present[t] = false;
        std::memset(p_.qt, 0, sizeof(p_.qt));
        p_.features &= ~kFeatDqt16;
    };
    uint8_t other_sof = 0;   // a frame header this decoder (like the reference: parser.cpp:82, SOF = 0xC0 only) does not handle
    while (!seen_sos) {
        if (p + 4 > len) return Fail("truncated before SOS");
        while (p < len && d[p] == 0xFF) p++;                                        // parser.cpp:75
        if (p + 3 > len) return Fail("truncated before SOS");
        uint8_t m = d[p++];
        uint32_t seglen = Rd16(d + p);
        size_t next = p + seglen;
        if (seglen < 2 || next > len) return Fail("bad segment length");
        const uint8_t* s = d + p;
        switch (m) {
            case 0xC0: if (!ParseSof(s, seglen, false)) return false; seen_sof0 = true; break;
            case 0xC1: if (!ParseSof(s, seglen, true)) return false; seen_sof0 = true; break;
            case 0xC2: case 0xC3: case 0xC5: case 0xC6: case 0xC7: case 0xC9: case 0xCA: case 0xCB: case 0xCD:
            case 0xCE: case 0xCF:
                other_sof = m;   // skipped by length as the reference does; the scan header then has no frame to refer to
                break;
            case 0xC4:
                if (!TakeTableSegment(dht_cache_, s + 2, seglen - 2, parse_dht, clear_dht)) return TablesFailed();
                seen_dht = true;
                break;
            case 0xDB:
                if (!TakeTableSegment(dqt_cache_, s + 2, seglen - 2, parse_dqt, clear_dqt)) return TablesFailed();
                seen_dqt = true;
                break;
            case 0xDD:                                                              // parser.cpp:374-390
                if (seglen != 4) return Fail("bad DRI length");
                p_.restart_interval = int32_t(Rd16(s + 2));
                break;
            case 0xDA:
                // same verdict as the reference (its ParseSOS finds no matching frame components, parser.cpp:340-358),
                // but say what the file is instead of reporting a component mismatch
                if (!seen_sof0 && other_sof) {
                    static const char* const kKind[16] = {"", "extended sequential", "progressive", "lossless", "", "differential sequential",
                                                          "differential progressive", "differential lossless", "", "arithmetic-coded sequential",
                                                          "arithmetic-coded progressive", "arithmetic-coded lossless", "", "arithmetic-coded differential",
                                                          "arithmetic-coded differential", "arithmetic-coded differential"};
                    const std::string why = std::string("not a baseline JPEG: ") + kKind[other_sof & 15] + " frame (SOF" +
                                            std::to_string(other_sof & 15) + ") - only baseline sequential DCT (SOF0) is decoded";
                    return Fail(why.c_str());   // Fail copies the text
                }
                if (!ParseSos(s, seglen)) return false;
                seen_sos = true;
                break;
            default: break;   // APPn, COM, SOF2 ... skipped by length (parser.cpp:105-108)
        }
        p = next;
    }
    if (!seen_dht) return Fail("no Huffman table before SOS");                     // parser.cpp:111-118
    if (!seen_dqt) return Fail("no quantisation table before SOS");
    if (!FinishTableSegments(dht_cache_, parse_dht, clear_dht) || !FinishTableSegments(dqt_cache_, parse_dqt, clear_dqt)) return TablesFailed();
    DeriveGeometry();
    p_.scan_offset = uint32_t(p);
    p_.raw_bytes = uint32_t(len - p);
    // restart intervals: what the frame needs, bounded by what the bytes can hold (a marker is two bytes)
    const uint64_t total_mcus = uint64_t(p_.mcus_x) * uint64_t(p_.mcus_y);
    const uint64_t by_header = (p_.restart_interval > 0 && total_mcus > 0) ? (total_mcus + uint64_t(p_.restart_interval) - 1) / uint64_t(p_.restart_interval) : 1;
    p_.nseg = uint32_t(std::min<uint64_t>(by_header, uint64_t(p_.raw_bytes) / 2 + 1));
    BuildDecodeTables();
    if (data_is_file_buffer) {   // already in this handle's page-locked memory: used in place
        raw_ = RawScan();
        raw_.nbytes = uint32_t(len - p);
        raw_.host = d + p;
        raw_.dev = file_.pinned() ? d + p : nullptr;
        if (raw_.dev) (void)DeviceAliasOf(d + p, &raw_.range_base, &raw_.range_size);
    } else {
        AdoptSource(d + p, len - p);
    }
    p_.valid = true;
    return true;
}

}  // namespace rjb
