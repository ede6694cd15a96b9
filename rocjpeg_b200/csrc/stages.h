// stages.h — host-callable launchers of the CUDA stages.
//
// These replace, for a whole batch per launch:
//   K0 (k0_destuff.cu)  the byte-serial FF D9 search of the reference's parser
//                       (src/rocjpeg_parser.cpp:400-416) and the destuffing / restart-marker
//                       handling VCN does on the slice it is given
//   K1 (k1_huffman.cu)  the Huffman decode done by VCN fixed function in the
//                       reference (src/rocjpeg_vaapi_decoder.cpp:677-689, 816-828)
//   K2 (k2_idct.cu)     the dequantise + IDCT done by VCN fixed function (same call sites);
//      (k2_scaled.cu)   its reduced-size forms for decodes at 1/2, 1/4 and 1/8 scale
//   K3 (k3_output.cu)   the post-processing kernels and copies of
//                       src/rocjpeg_hip_kernels.cpp / src/rocjpeg_decoder.cpp:372-636
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_types.h"

namespace rjb {

#ifdef __CUDACC__
// Programmatic dependent launch: consecutive kernels of a lane's stream are chained so that a kernel's
// CTAs are placed and run their prologue while the previous kernel's last CTAs drain, instead of paying a
// full launch latency at every one of the dozen stage boundaries (the single-picture decode is made of
// them). Every kernel starts with PdlEntry(): it waits until its predecessor has completed and its writes
// are visible - stream order is preserved exactly. Measured on c3 / c2: 0.597 -> 0.538 ms and 0.220 ->
// 0.188 ms per batch. Triggering the successor EARLY (griddepcontrol.launch_dependents at kernel entry,
// RJB_PDL_TRIGGER=1) parks its CTAs, shared memory included, on the SMs while they wait: with several
// pipeline lanes that takes occupancy from the other lanes' running kernels (c3: 0.669 ms) - left off.
#ifndef RJB_PDL_TRIGGER
#define RJB_PDL_TRIGGER 0
#endif
__device__ __forceinline__ void PdlEntry() {
#if RJB_PDL_TRIGGER
    asm volatile("griddepcontrol.launch_dependents;");
#endif
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <class... KArgs, class... Args>
inline cudaError_t LaunchPdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

constexpr int kK0TileBytes = 16384;  // raw bytes per destuffing tile (one CTA, 64 bytes per thread) = bytes per gather step
constexpr int kK1Threads = 128;      // threads per CTA in K1, one subsequence each
constexpr int kDcImageMaxMcus = 4096;   // pictures up to this many MCUs take the one-launch DC integration
// K1Args::halo leading threads of a CTA re-decode the previous CTA's last subsequences; the CTA owns the
// kK1Threads - halo subsequences behind them (chosen per batch, decoder.cpp)
constexpr int kDcTileMcus = 256;     // MCUs per DC-scan tile
constexpr int kMaxSyncRounds = 8;    // counters kept per batch
constexpr int kK3TileW = 256;        // output tile of the colour/layout stage, in luma samples
constexpr int kK3TileH = 32;
constexpr uint32_t kNoEntry = 0xFFFFFFFFu;   // BlockRec::end of a block no thread reached (damaged streams)

// What K1 leaves per 8x8 block besides its coefficient entries (decode order, filled with 0xFF
// before every decode): where its entries end — they begin where the previous block's end,
// block 0 of an image at entry 0 — and its DC value: the difference after k1_write, the
// integrated DC after dc_apply.
struct BlockRec {
    uint32_t end;   // index one past the block's last entry, relative to the image's stream
    int16_t dc;
    int16_t pad_;
};

struct K0Args {
    const ImageDesc* images;      // device
    SegmentDesc* segments;        // device, written here: the batch's segment table
    const uint32_t* img_tile0;    // device, nimages + 1 entries: first destuffing tile of each image
    const uint8_t* raw;           // device raw arena (bytes as uploaded)
    uint8_t* clean;               // device scan arena (destuffed)
    uint4* tile_sum;              // per tile: prefix element of the tile
    uint4* tile_carry;            // per tile: prefix element of everything before it in its image
    ScanStatus* status;           // per image
    int nimages;
    uint32_t total_tiles;
    int sub_bytes;                // S of the batch: intervals start on multiples of S
    int inline_scan;              // no image has more than 32 tiles: k0_apply combines the earlier tiles' elements itself, no k0_scan
};
// Gather per-image raw bytes from mapped page-locked host memory into the raw arena.
struct GatherItem {
    const uint8_t* src;   // device-visible address of the 16-byte vector the image's first entropy-coded byte lies in
    uint64_t dst_off;     // byte offset in the raw arena
    uint32_t nbytes;      // multiple of 16
    uint32_t pad_;
};
// Per-tile prefix elements of the raw bytes already in the arena (cudaMemcpy uploads, resident re-runs) ...
cudaError_t LaunchK0Reduce(const K0Args& a, cudaStream_t stream);
// ... or computed on the way by the kernel that uploads them (items: device array, one per image).
cudaError_t LaunchGatherReduce(const K0Args& a, const GatherItem* items, cudaStream_t stream);
// Scan over the tiles + scatter: destuffed bytes, restart intervals, segment table (two launches).
cudaError_t LaunchK0Destuff(const K0Args& a, cudaStream_t stream);
cudaError_t PreloadK0();

struct K1Args {
    const ImageDesc* images;      // device
    const SegmentDesc* segments;  // device
    const uint32_t* img_cta0;     // device, nimages + 1 entries: first K1 CTA of each image
    const uint32_t* img_dctile0;  // device, nimages + 1 entries: first DC tile of each image
    const uint8_t* scan;          // device scan arena
    const HuffLutSet* luts;       // device
    uint32_t* state;              // per subsequence: packed out-state | blocks << 16
    uint32_t* used;               // per subsequence: key of the in-state its state was decoded from
    uint32_t* sub_seg;            // per subsequence: segment index (cache)
    uint32_t* nnz;                // per subsequence: coefficient entries it produces
    uint2* cta_partial;           // per K1 CTA: (has segment start, blocks after the last start)
    uint32_t* cta_entries;        // per K1 CTA: coefficient entries of the CTA's subsequences
    uint2* cta_carry;             // per K1 CTA: (blocks, entries) entering it from the image's earlier CTAs (k1_scan)
    uint32_t* cta_flag;           // per K1 CTA: k1_fused has published the CTA's counts and states (1) and written its records (2);
                                  // [total_ctas] = its ticket counter; [total_ctas + 1 + k] = CTA k has published its DC sums (1) and
                                  // the predictors leaving it (2) (all zeroed before the launch)
    int4* cta_dc;                 // per K1 CTA (k1_fused with k1_dc): [2 k] per-component DC sums of its block range after its last
                                  // predictor reset (.w: the range holds one), [2 k + 1] predictors leaving it
    int3* dc_partial;             // per DC tile: per-component DC sum after the tile's last reset
    int3* dc_carry;               // per DC tile: predictors entering it (dc_scan)
    uint32_t* counters;           // [kMaxSyncRounds] boundary changes per round, then [kMaxSyncRounds] decodes per round
    uint32_t* counters_next;      // the next batch's set (64 words): k1_write zeroes it
    ScanStatus* status;           // per image: the write pass ORs kDecodeShort into the flags
    uint32_t* entries;            // coefficient entry arena (huff_core.cuh: MakeCoefEntry), decode order
    BlockRec* blk_rec;            // per block, decode order
    int nimages;
    uint32_t total_ctas;          // K1 CTAs in the batch
    uint32_t total_dc_tiles;
    int sub_bytes;                // subsequence size S in bytes: 32, 64 or 128
    uint32_t lut_smem_bytes;      // shared memory for the Huffman tables: 4 KiB per table pair + the second-level arena (batch maximum)
    uint32_t rec_fill_vecs;       // 16-byte vectors of blk_rec that round 0 of k1_sync fills with 0xFF ("never decoded")
    int halo;                     // threads of a CTA that re-decode the subsequences before the CTA's own
    int inline_scan;              // no image has more than 32 K1 CTAs: k1_write sums the partials of the image's earlier CTAs
                                  // itself (one warp, one load each) and k1_scan is not launched
    int fusable;                  // no image has more than 256 K1 CTAs: counting and write pass may run as one kernel (k1_fused)
    int dc_image;                 // no image has more than kDcImageMaxMcus MCUs: one CTA per image integrates its DC
                                  // differences in ONE launch (dc_image) instead of sums / scan / apply
    int k1_dc;                    // k1_fused integrates the DC differences itself: LaunchDcScan is not needed after it
};

// Speculative decode + CTA-local synchronisation (round 0) or cross-CTA fix-up (round >= 1).
// max_iters bounds the CTA-local fix-up loop (<= 0: until nothing changes).
cudaError_t LaunchK1Sync(const K1Args& a, int round, cudaStream_t stream, int max_iters = 0);
// Final pass: positions from the block counts, coefficients and DC differences written.
cudaError_t LaunchK1Write(const K1Args& a, cudaStream_t stream);
// Both in one kernel (batches whose pictures have at most 256 K1 CTAs, K1Args::fusable); counters[0] = CTA boundaries whose
// handed-over state was not the owner's: non-zero -> run LaunchK1Sync rounds >= 1 and LaunchK1Write.
cudaError_t LaunchK1Fused(const K1Args& a, cudaStream_t stream);
cudaError_t LaunchK1ClearShort(const K1Args& a, cudaStream_t stream);   // before that fallback's LaunchK1Write
// DC prediction: per-tile sums, then prefix; absolute DC written over the per-block differences.
cudaError_t LaunchDcScan(const K1Args& a, cudaStream_t stream);

struct K2Args {
    const ImageDesc* images;
    const OutputDesc* outputs;    // for images whose planes go straight to the caller's buffers (OutputDesc::direct)
    int force_planes;             // 1: ignore `direct`, write the plane arena (stage tap)
    const uint32_t* img_tile0;    // nimages + 1: first IDCT tile of each image
    const uint16_t* qtables;      // natural-order u16[64] tables
    const uint32_t* entries;      // coefficient entries
    const BlockRec* blk_rec;      // end-of-entries index + integrated DC of every block (decode order)
    uint8_t* planes;              // plane arena
    int nimages;
    uint32_t total_tiles;
};
cudaError_t LaunchK2Idct(const K2Args& a, cudaStream_t stream);
// Reduced-size IDCT (k2_scaled.cu) for the pictures decoded at scale 1 / scale_denom (2, 4 or 8): every block yields an
// (8 / scale_denom)-sample square. Same tiles and arguments as LaunchK2Idct; planes, pitches, crop rectangle and the
// caller's channels are in scaled units.
cudaError_t LaunchK2Scaled(const K2Args& a, int scale_denom, cudaStream_t stream);

// K2 + K3 in one kernel for whole-picture RGB / RGB_PLANAR outputs (OutputDesc::fused): coefficients in, pixels out.
struct K23Args {
    const FusedImage* fused;      // one per image served by this kernel
    const uint32_t* tile_img;     // per strip of k23_fused (pictures with unaligned destination rows): index into `fused` | MCU row << 16
    const uint32_t* tile_img_w;   // per strip of k23_warp (destination rows 4-byte aligned), same encoding
    const uint16_t* qtables;
    const uint32_t* entries;
    const BlockRec* blk_rec;
    int nimages;
    uint32_t total_tiles, total_tiles_w;
};
cudaError_t LaunchK23Fused(const K23Args& a, cudaStream_t stream);
cudaError_t PreloadK23();

struct K3Args {
    const ImageDesc* images;
    const OutputDesc* outputs;
    const uint32_t* img_tile0;    // nimages + 1: first output tile of each image
    const uint8_t* planes;
    int nimages;
    uint32_t total_tiles;
};
cudaError_t LaunchK3Output(const K3Args& a, cudaStream_t stream);

// Load the stages' kernels now instead of at their first launch.
cudaError_t PreloadK1();
cudaError_t PreloadK2();
cudaError_t PreloadK2Scaled();
cudaError_t PreloadK3();

}  // namespace rjb
