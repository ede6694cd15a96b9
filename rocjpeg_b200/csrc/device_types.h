// device_types.h — plain structs shared by the host orchestrator and the CUDA stages.
//
// Nothing here exists in the reference: its Huffman/IDCT stage is the VCN
// fixed-function block behind libva (src/rocjpeg_vaapi_decoder.cpp:677-689).
// These descriptors are what replaces the five VA buffers of one picture
// (picture / IQ matrix / Huffman / slice parameter / slice data) when the same
// work is done by sm_100a kernels over a whole batch in one launch per stage.
#pragma once
#include <stdint.h>

#ifndef __CUDACC__
#ifndef __host__
#define __host__
#define __device__
#endif
#endif

namespace rjb {

constexpr int kMaxBlocksPerMcu = 10;   // T.81 B.2.3
constexpr int kFastBits = 9;           // first-level Huffman LUT width
constexpr int kFastSize = 1 << kFastBits;
constexpr int kSubCap = 1024;          // second-level entries shared by the four tables of a set

enum Css : int32_t { CSS_444 = 0, CSS_440 = 1, CSS_422 = 2, CSS_420 = 3, CSS_411 = 4, CSS_400 = 5, CSS_UNKNOWN = -1 };
enum Fmt : int32_t { FMT_NATIVE = 0, FMT_YUV_PLANAR = 1, FMT_Y = 2, FMT_RGB = 3, FMT_RGB_PLANAR = 4 };

constexpr int kHuffIds = 4;            // Huffman table ids per class (T.81 B.2.4.2: Th 0..3; baseline files use 0 and 1)
constexpr int kHuffTabs = 2 * kHuffIds;   // slots of a set: 0..3 = DC tables 0..3, 4..7 = AC tables 0..3

// One set of Huffman tables (slot t < kHuffIds = DC table t, slot kHuffIds + t = AC table t), decoder form: a two-level
// lookup over 32-bit entries (huff_core.cuh: MakeEntry / MakeLink).
//   fast[t][next 9 bits]  symbol entry when the code is at most kFastBits long, else a link to a
//                         sub-table in `sub` indexed by the following x bits (x = longest code under
//                         that prefix - kFastBits), else (sub arena exhausted by a pathological
//                         table) a link with x = 0: the canonical search below resolves the code.
//   canonical search (T.81 F.2.2.3 restated left-aligned): first l in (kFastBits,16] with
//   peek16 < upper[t][l] has length l and symbol vals[t][(peek16 >> (16-l)) + valoff[t][l]].
// K1 stages fast + the used part of sub in shared memory; upper/valoff/vals stay in global memory.
struct HuffLutSet {
    uint32_t fast[kHuffTabs][kFastSize];
    uint32_t sub[kSubCap];
    uint32_t sub_used;       // entries of `sub` in use
    uint32_t pad_[3];
    uint32_t upper[kHuffTabs][17];   // exclusive upper bound of codes of length l, left-aligned to 16 bits
    int32_t valoff[kHuffTabs][17];   // valptr[l] - mincode[l]
    uint8_t vals[kHuffTabs][256];
};

// Geometry + bookkeeping of one image inside a batch (device-resident array).
struct ImageDesc {
    int32_t width, height, ncomp, css;
    int32_t mcus_x, mcus_y, bpm, restart_interval;   // bpm = blocks per MCU
    int32_t total_mcus;
    int32_t hs[3], vs[3];
    int32_t blocks_w[3], blocks_h[3];                 // MCU-padded block grid per component
    int32_t comp_first_blk[3];                        // index of a component's first block inside the MCU
    uint8_t mcu_comp[kMaxBlocksPerMcu];               // block-in-MCU -> component
    uint8_t mcu_dc[kMaxBlocksPerMcu];                 // block-in-MCU -> DC table slot in HuffLutSet
    uint8_t mcu_ac[kMaxBlocksPerMcu];                 // block-in-MCU -> AC table slot in HuffLutSet (kHuffIds + id)
    uint8_t mcu_pair[kMaxBlocksPerMcu];               // block-in-MCU -> table pair (index into pair_dc / pair_ac)
    uint8_t npairs;                                   // distinct (DC table, AC table) pairs the scan uses: 1..3
    uint8_t pair_dc[3], pair_ac[3];                   // HuffLutSet slot of each pair's DC / AC table
    uint8_t pad_[3];
    int32_t lut_set;                                  // index into the batch's HuffLutSet array
    int32_t qt_index[3];                              // index into the batch's quant-table array (natural order u16[64])
    // entropy-coded data as uploaded (raw: byte stuffing, fill bytes and restart markers still in it)
    uint64_t raw_off;                                 // byte offset of the image's raw bytes in the raw arena (16-byte aligned)
    uint32_t raw_skip;                                // bytes in front of the first entropy-coded byte (0..15: whole 16-byte vectors are uploaded)
    uint32_t raw_len;                                 // entropy-coded bytes present, up to the end of the caller's buffer (the slice ends at the first FF D9)
    uint32_t k0_tile0;                                // first destuffing tile of this image
    uint32_t seg_keep_lo, seg_keep_hi;                // restart intervals to decode, inclusive (region of interest; otherwise 0 .. nseg - 1)
    // entropy-coded data destuffed by k0 (restart interval k starts at clean offset SegmentStart(r_k, k, S), see below)
    uint64_t data_off;                                // byte offset of the image's clean stream in the scan arena (128-byte aligned)
    uint32_t seg0, nseg;                              // this image's slice of the batch segment table
    uint32_t sub0, nsub;                              // first subsequence (multiple of the CTA size) and count: clean capacity / S
    // coefficient store: a sparse stream of (int16 value, zig-zag index) entries in decode order
    // plus one record per block {where its entries end, DC} (stages.h: BlockRec)
    uint64_t blk0;                                    // first block of this image in the per-block arrays
    uint64_t ent0;                                    // first entry of this image in the entry arena
    uint32_t ent_cap;                                 // entries reserved for this image (upper bound from the scan size)
    uint32_t nblocks;
    uint32_t dc_tile0;                                // first DC-scan tile of this image
    uint32_t comp_bits;                               // mcu_comp packed, two bits per block-in-MCU (the DC kernels unroll over it)
    // decoded component planes (MCU-padded), u8
    uint64_t plane_off[3];
    uint32_t plane_pitch[3];
};

// Where restart interval k of an image starts in the image's clean stream, as a function of where its
// bytes start in the RAW stream (r = raw position just behind the k-th restart marker, 0 for k = 0) -
// so that the destuffing pass can place every interval without knowing the lengths of the others.
// Destuffing only removes bytes, an interval's clean length n_k is at most r_{k+1} - 2 - r_k, hence
//   Start(k+1) - Start(k) >= (r_{k+1} - r_k) + S + 14 - (S - 1) >= n_k + 17:
// intervals never overlap, start on a subsequence boundary (multiple of S) and leave room for the 16 zero
// bytes the bit reader may look ahead into. Subsequence g of the image covers clean bytes [g S, (g+1) S).
__host__ __device__ inline uint64_t SegmentStart(uint32_t r, uint32_t k, uint32_t S) {
    return (uint64_t(r) + uint64_t(S + 14u) * k + (S - 1u)) / S * S;
}
// Clean-stream capacity of an image with `raw_len` raw bytes and at most `nseg` restart intervals.
__host__ __device__ inline uint64_t CleanCapacity(uint32_t raw_len, uint32_t nseg, uint32_t S) {
    return (SegmentStart(raw_len, nseg, S) + S + 127u) / 128u * 128u;
}

// Per-image outcome of the destuffing pass (device -> host with the status read-back).
struct ScanStatus {
    uint32_t segments_seen;   // restart intervals found in the bytes (restart markers + 1)
    uint32_t scan_size;       // raw bytes up to the first FF D9 (= raw_len when there is none)
    uint32_t flags;           // kScan* (destuffing pass) | kDecode* (entropy stage); OR-ed in by many threads, zeroed by the tile reduction
    uint32_t reserved;
};
constexpr uint32_t kScanNoEoi = 1u,            // no FF D9: the slice ran to the end of the buffer
                   kScanStrayMarker = 2u,      // a marker other than RSTn / EOI inside the entropy-coded data
                   kScanExtraRestarts = 4u,    // more restart markers than the frame has restart intervals
                   kScanMissingIntervals = 8u, // fewer restart intervals in the bytes than the frame needs (set on the host)
                   kScanEmptyInterval = 16u,   // a restart interval that must hold blocks holds no bytes
                   kDecodeShort = 32u;         // a restart interval ran out of bytes before its last block
constexpr uint32_t kStatusTruncatedMask = kScanMissingIntervals | kScanEmptyInterval | kDecodeShort;   // -> BAD_JPEG

// One restart interval ("segment") of one image: an independently decodable,
// byte-aligned run of entropy-coded data with predictors reset (T.81 E.1.4).
// Written by the destuffing pass (k0_destuff.cu), never by the host.
struct SegmentDesc {
    uint64_t data_off;     // byte offset in the scan arena (16-byte aligned)
    uint32_t nbytes;       // entropy-coded bytes in the segment (excludes padding)
    uint32_t sub0;         // first subsequence of the segment (global index)
    uint32_t blk_first;    // first block of the segment, relative to the image's blk0
    uint32_t blk_count;    // blocks the segment must produce (MCUs in interval * bpm)
};

// Output job for the colour/layout stage: one destination image.
struct OutputDesc {
    uint8_t* dst[4];
    uint32_t dst_pitch[4];
    int32_t x0, y0, w, h;    // region of interest in luma samples (whole picture when no crop)
    int32_t fmt;
    uint32_t tile0;          // first output tile of this image
    uint32_t tiles_x, tiles_y;
    int32_t direct;          // the IDCT stage stores this image's planes straight into dst (planar formats, no crop): no output tiles
    int32_t fused;           // whole-picture RGB / RGB_PLANAR: the fused IDCT + output kernel serves it (no IDCT tiles' output, no output tiles)
    int32_t jfif;            // RGB / RGB_PLANAR under the libjpeg colour convention: k3_jfif serves it, and a crop needs the chroma around it
    int32_t upsample;        // UpsampleMode of k3_jfif
    int32_t pic_w, pic_h;    // the picture's size at its scale (the crop rectangle lies inside it): the upsampling's edges
};

// Chroma upsampling of k3_jfif.cu: the method libjpeg-turbo's jinit_upsampler (jdsample.c) picks for the component ratio.
enum UpsampleMode : int32_t { UP_REPLICATE = 0, UP_H2V1 = 1, UP_H1V2 = 2, UP_H2V2 = 3 };

// Everything the fused IDCT + output kernel (k23_fused.cu) needs about one picture, prepared on the host so that a CTA
// starts from one record instead of deriving it (a quarter of the kernel's time when thread 0 did: profiles/r02_*).
struct FusedImage {
    uint64_t ent0, blk0;          // the picture's coefficient entries / block records
    uint8_t* dst[3];
    uint32_t dpitch;              // pitch[0]: RGB rows, and all three RGB_PLANAR planes (src/rocjpeg_decoder.cpp:526-544)
    uint32_t ent_cap;
    int32_t width, height, css, fmt;
    int32_t ncomp, bpm, mcus_x, vmax;
    int32_t mpt;                  // MCUs per 256-sample strip
    uint32_t tiles_x;             // strips per MCU row
    uint32_t tile0;               // first strip of the picture
    int32_t sx, sy;               // chroma shifts
    uint8_t H[3], V[3], first_blk[3], hshift[3];
    uint32_t qidx[3];             // quantiser table per component
    uint32_t pitch[3], base[3];   // shared-memory plane pitch / offset per component
    uint32_t comp_info[3];        // H | V << 8 | first_blk << 16 | hshift << 24: one load per component in k23_warp
};

}  // namespace rjb
