// jpeg_parser.h — host-side baseline JPEG stream parser.
//
// Behaviour-compatible replacement for the reference's RocJpegStreamParser
// (src/rocjpeg_parser.h:180-269, src/rocjpeg_parser.cpp): same marker walk and
// the same accept/reject decisions (SOF0 only, <=3 components, 8-bit DQT with
// id<4, DHT id<2, SOS ids must follow SOF order, DRI length 4, at least one DHT
// and one DQT before SOS, entropy-coded slice = bytes up to the first FF D9),
// plus bounds checks (the reference reads past the end of truncated input).
//
// Extended for the CUDA back end (BASELINE north star, item 2). Parsing costs a
// header walk, nothing proportional to the picture:
//   * the entropy-coded bytes are NOT touched on the host. The reference makes one
//     byte-serial pass over them to find FF D9 (src/rocjpeg_parser.cpp:400-416);
//     here that pass - together with the removal of byte stuffing (FF 00 -> FF),
//     fill bytes and restart markers and the discovery of the restart intervals -
//     runs on the GPU (k0_destuff.cu), on the raw bytes as uploaded. The parser only
//     makes the bytes reachable by the device: a caller buffer that is already
//     page-locked (cudaHostAlloc / cudaHostRegister / hipHostMalloc through the
//     shim) is used in place, anything else is copied once into page-locked
//     staging taken from a process-wide pool;
//   * it builds the decoder-form Huffman tables (two-level LUT + canonical slow
//     path) and natural-order quantisation tables.
// The host restatement of the same destuffing rules (HostScan) is kept for the
// parser taps, the K1 schedule model and as the expected value of the GPU pass in
// the tests; the decode path never calls it.
#pragma once
#include <cstddef>
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "device_types.h"

namespace rjb {

// ROCJPEG_B200_POISON=<byte> (test knob; decimal or 0x..): every device arena and every grant of page-locked staging is
// filled with that byte before first use, so that a kernel reading memory no call wrote shows in the output instead of
// finding cudaMalloc's zeros or an earlier call's values. -1 when unset. Read at each allocation, so a test can set it
// before creating a handle.
int PoisonByte();

// Grow-only host buffer; page-locked (cudaHostAlloc, portable + mapped) when a
// CUDA driver is present, plain aligned memory otherwise (CPU-only unit tests).
class StagingBuffer {
  public:
    StagingBuffer() = default;
    ~StagingBuffer();
    StagingBuffer(const StagingBuffer&) = delete;
    StagingBuffer& operator=(const StagingBuffer&) = delete;
    uint8_t* Reserve(size_t bytes);   // contents are NOT preserved across growth
    uint8_t* data() const { return ptr_; }
    size_t capacity() const { return cap_; }
    bool pinned() const { return pinned_; }

  private:
    void Release();
    uint8_t* ptr_ = nullptr;
    size_t cap_ = 0;
    bool pinned_ = false;
};

// Process-wide pool of page-locked host memory (cudaHostAlloc, portable + mapped) handed out in
// power-of-two blocks: stream handles that receive pageable input stage it here. One slab
// allocation serves hundreds of handles (a cudaHostAlloc per handle was 32 ms for 256 handles).
class PinnedPool {
  public:
    static PinnedPool& Get();
    // Returns a block of at least `bytes` (capacity in *cap); pageable memory when no CUDA driver
    // is present (*pinned = false; host-only unit tests).
    uint8_t* Alloc(size_t bytes, size_t* cap, bool* pinned);
    void Free(uint8_t* p, size_t cap, bool pinned);

  private:
    PinnedPool() = default;
    std::mutex m_;
    std::vector<std::vector<uint8_t*>> free_;   // by size class (log2)
    uint8_t* slab_ = nullptr;
    size_t slab_left_ = 0, next_slab_ = 0;
    bool no_driver_ = false;
};

// Grow-only block from the pool.
class PooledBuffer {
  public:
    PooledBuffer() = default;
    ~PooledBuffer() { Release(); }
    PooledBuffer(const PooledBuffer&) = delete;
    PooledBuffer& operator=(const PooledBuffer&) = delete;
    uint8_t* Reserve(size_t bytes);   // contents are NOT preserved across growth
    void Release();
    uint8_t* data() const { return ptr_; }
    bool pinned() const { return pinned_; }

  private:
    uint8_t* ptr_ = nullptr;
    size_t cap_ = 0;
    bool pinned_ = false;
};

// What a stream may use beyond the reference's parser (SURVEY.md section 8 f4): SOF1 with 8-bit samples (the same decode
// process as SOF0; libjpeg-turbo writes it as soon as a quantiser step exceeds 255), 16-bit quantiser steps (rejected at
// src/rocjpeg_parser.cpp:230) and Huffman table ids 2 and 3 (rejected at :274).
constexpr int32_t kFeatSof1 = 1, kFeatDqt16 = 2, kFeatHuffId23 = 4;

struct HuffSpec {
    uint8_t bits[16];
    uint8_t vals[256];
    uint32_t count;
    bool present;
};

struct Segment {
    uint32_t offset;   // byte offset inside the clean stream (16-byte aligned)
    uint32_t nbytes;   // entropy-coded bytes
};

// Everything one parsed picture contributes to a decode call.
struct ParsedJpeg {
    bool valid = false;
    // frame / scan header (field-for-field what the reference keeps in
    // JpegStreamParameters, src/rocjpeg_parser.h:150-172)
    int32_t width = 0, height = 0, ncomp = 0, css = CSS_UNKNOWN;
    int32_t comp_id[3] = {0, 0, 0}, hs[3] = {0, 0, 0}, vs[3] = {0, 0, 0}, tq[3] = {0, 0, 0};
    int32_t scan_ncomp = 0, td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
    int32_t restart_interval = 0;
    uint32_t num_mcus_ref = 0;                    // the reference's num_mcus (parser.cpp:197)
    uint32_t scan_offset = 0;                     // first entropy-coded byte inside the caller's buffer (parser.cpp:400-416)
    uint32_t raw_bytes = 0;                       // from there to the end of the caller's buffer (the slice ends at the first
                                                  // FF D9, which the GPU pass finds; HostScan::scan_size on the host)
    uint16_t qt[4][64] = {};                      // zig-zag order, as in the stream (8- or 16-bit steps)
    bool qt_present[4] = {false, false, false, false};
    HuffSpec dc[kHuffIds] = {}, ac[kHuffIds] = {};
    int32_t features = 0;                         // kFeat*: what the stream uses beyond what the reference's parser accepts
    // derived geometry (T.81 A.1.1, A.2)
    int32_t hmax = 1, vmax = 1, mcus_x = 0, mcus_y = 0, bpm = 0;
    int32_t blocks_w[3] = {0, 0, 0}, blocks_h[3] = {0, 0, 0};
    // decode-side products
    int32_t support_status = 0;                   // RocJpegStatus value: 0 when the CUDA path can decode it
    uint16_t qt_natural[4][64] = {};              // de-zig-zagged quantiser steps
    uint64_t lut_hash = 0;                        // identity of the four Huffman tables (batch de-duplication)
    uint32_t min_entry_bits = 2;                  // fewest bits a symbol with magnitude bits can take (bounds the entry count)
    uint32_t nseg = 1;                            // restart intervals the scan can hold: ceil(mcus / Ri), bounded by the bytes present
};

// Where the entropy-coded bytes of the last parsed stream are, for the upload.
struct RawScan {
    const uint8_t* host = nullptr;   // first entropy-coded byte: inside the caller's buffer (zero-copy) or the handle's staging
    const uint8_t* dev = nullptr;    // the same byte as the device sees it (page-locked memory); nullptr: pageable, copy with cudaMemcpy
    uint32_t nbytes = 0;
    bool zero_copy = false;          // `host` is the caller's own page-locked buffer
    // the page-locked allocation `host` lies in (0, 0: unknown): streams of one allocation that lie close together
    // are uploaded with one copy (decoder.cpp: Lane::Build)
    uintptr_t range_base = 0;
    size_t range_size = 0;
};

// Host restatement of the destuffing pass (tests, taps, schedule model - never the decode path).
struct HostScan {
    bool done = false;
    uint32_t scan_size = 0;                       // bytes up to the first FF D9 (the reference's slice size)
    uint32_t restart_markers_seen = 0;
    std::vector<Segment> segments;                // one per restart interval (exactly ParsedJpeg::nseg)
    std::vector<uint8_t> clean;                   // destuffed bytes, 16-byte-aligned segments, zero padded
    size_t clean_bytes = 0;
};

class StreamParser {
  public:
    // Returns false for streams the reference parser rejects (-> BAD_JPEG).
    bool Parse(const uint8_t* data, size_t length);
    // File -> device ingestion (the step before the path in the reference's samples: an ifstream read per image on the
    // decode thread, samples/rocjpeg_samples_utils.h:213-234): the file is read straight into this handle's pooled
    // page-locked staging and parsed there - no intermediate copy, the upload reads the staging in place.
    // Returns 0, -2 (cannot open / read: see last_error), -3 (not a JPEG this parser accepts).
    int ParseFile(const char* path);
    const ParsedJpeg& parsed() const { return p_; }
    const RawScan& raw() const { return raw_; }
    // Pageable input is copied into page-locked staging by Parse() - or, with ROCJPEG_B200_DEFERRED_COPY=1, when the decode
    // call needs the bytes (by its helper threads, several streams at a time, chunk by chunk alongside the uploads; the
    // caller's buffer is then borrowed from rocJpegStreamParse until the decode returns, as the reference requires:
    // src/rocjpeg_parser.cpp:413 keeps a pointer into it). EnsureStaged is idempotent; a second decode finds the copy.
    bool staging_pending() const { return pending_src_ != nullptr; }
    void EnsureStaged() const;
    // Destuffed restart intervals computed on the host from the bytes Parse() was given (which must still
    // be valid, as the reference requires until the decode returns).
    const HostScan& host_scan() const;
    const HuffLutSet& lut() const { return lut_ ? *lut_ : EmptyLut(); }   // decoder-form tables of the last parsed stream
    const std::string& last_error() const { return err_; }

  private:
    bool Fail(const char* why);
    bool ParseSof(const uint8_t* s, uint32_t seglen, bool extended);
    bool ParseDht(const uint8_t* payload, uint32_t n);   // payload = the segment behind its two length bytes
    bool ParseDqt(const uint8_t* payload, uint32_t n);
    bool ParseSos(const uint8_t* s, uint32_t seglen);
    void DeriveGeometry();
    void ExtractEntropyData(const uint8_t* d, size_t length, HostScan* out) const;
    void BuildDecodeTables();
    void AdoptSource(const uint8_t* scan, size_t nbytes);
    void EnsureStagedLocked() const;
    bool ParseLocked(const uint8_t* data, size_t length, bool data_is_file_buffer);
    void ResetFrame();
    // Table segments (DHT / DQT) of the stream being parsed against the previous stream's: while the payload bytes
    // repeat - the normal case, the same encoder wrote the files - nothing is re-parsed, re-hashed or rebuilt.
    struct TableCache {
        std::vector<uint8_t> key;                           // payloads of the previous stream's segments, concatenated
        size_t cursor = 0;                                  // bytes of `key` matched so far
        bool matching = false;                              // every segment so far repeated the previous stream's
        bool changed = false;                               // the tables were re-parsed during this Parse()
        const uint8_t* seg[8] = {};                         // this stream's segments (payload pointers / lengths) ...
        uint32_t seglen[8] = {};
        int nseg = 0;                                       // ... more than 8: no caching
        void Begin() { cursor = 0; matching = !key.empty(); changed = false; nseg = 0; }
    };
    template <class ParseFn, class ClearFn> bool TakeTableSegment(TableCache& c, const uint8_t* payload, uint32_t n, ParseFn parse, ClearFn clear);
    template <class ParseFn, class ClearFn> bool FinishTableSegments(TableCache& c, ParseFn parse, ClearFn clear);
    TableCache dht_cache_, dqt_cache_;

    mutable std::mutex mutex_;
    ParsedJpeg p_;
    // Decoder-form tables: shared with the process-wide cache (jpeg_parser.cpp: BuildDecodeTables) - a handle holds a
    // reference, not 22 KiB of its own (creating 256 handles spent 3 ms faulting those pages in).
    std::shared_ptr<const HuffLutSet> lut_;
    static const HuffLutSet& EmptyLut();
    uint32_t lut_cap_ = 0;
    bool lut_valid_ = false;
    bool TablesFailed();              // a table segment was rejected: nothing of it may be reused by the next parse
    RawScan raw_;
    mutable const uint8_t* pending_src_ = nullptr;   // pageable source not yet copied into staging_ (EnsureStaged)
    mutable size_t pending_len_ = 0;
    PooledBuffer staging_;            // page-locked copy of pageable input
    PooledBuffer file_;               // a whole file read by ParseFile (page-locked)
    mutable HostScan host_scan_;
    std::string err_;
};

int ClassifyChromaSubsampling(const int32_t h[3], const int32_t v[3]);
void BuildHuffLut(const HuffSpec& spec, int slot, HuffLutSet* out, uint32_t sub_cap = kSubCap);

}  // namespace rjb
