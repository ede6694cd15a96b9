/* rocjpeg_b200_ext.h — extension entry points of the B200-native librocjpeg.so.
 *
 * The drop-in boundary is include/rocjpeg.h (the reference's api/rocjpeg.h,
 * unchanged). The functions below are ADDITIONS used by this repository's
 * parity tests and bench.py; nothing in the reference binds them:
 *   - stage taps, so that the intermediate results the reference never exposes
 *     (they live inside the VCN engine, src/rocjpeg_vaapi_decoder.cpp:677-689)
 *     can be compared with the oracle: quantised coefficients (vs libjpeg-turbo
 *     jpeg_read_coefficients) and decoded component planes (vs jpeg_read_raw_data);
 *   - a split prepare/run form of rocJpegDecodeBatched (api/rocjpeg.h:331) so the
 *     device-resident throughput ("inputs already in HBM") can be timed apart
 *     from the host->device copy;
 *   - decodes at 1/2, 1/4 and 1/8 scale (reduced-size IDCT, as libjpeg's scale_denom);
 *   - decodes resized to a requested size as Pillow's Image.resize does it;
 *   - per-stage CUDA-event timings and batch statistics for the roofline report;
 *   - parser taps (host only; usable without a GPU).
 * Plain C ABI: pointers and sizes only.
 */
#ifndef ROCJPEG_B200_EXT_H
#define ROCJPEG_B200_EXT_H

#include <stddef.h>
#include <stdint.h>

#include "rocjpeg.h"

#if defined(__cplusplus)
extern "C" {
#endif

#define ROCJPEG_B200_STAGE_COUNT 7 /* upload, destuff, huffman-sync (the whole entropy stage when it runs as one kernel), huffman-write, dc, idct,
                                      output (the fused IDCT + output kernels included) */

typedef struct {
    float stage_ms[ROCJPEG_B200_STAGE_COUNT]; /* CUDA-event time of each stage on the decoder's stream */
    float total_ms;                           /* first to last event */
    uint32_t sync_rounds;                     /* 1: the fused entropy kernel alone (k1_fused, its CTA-boundary check held); else k1_sync
                                                 launches (2 when the stream self-synchronises within the counting + verifying round) */
    uint32_t decodes_per_round[8];            /* subsequence decodes performed in each round */
    uint64_t scan_bytes;                      /* entropy-coded bytes of the batch as uploaded (before destuffing) */
    uint64_t blocks;                          /* 8x8 blocks decoded */
    uint64_t subsequences;
    uint64_t plane_bytes;                     /* component-plane bytes written by the IDCT stage */
    uint64_t output_bytes;                    /* bytes written to the caller's buffers */
    uint64_t h2d_bytes, d2h_bytes;            /* host<->device traffic of the last call */
    uint32_t kernel_launches;                 /* kernels launched by the last call */
    int32_t subsequence_bytes;                /* S chosen for the batch */
    int32_t lanes;                            /* pipeline lanes (streams) the batch was split over */
    float host_submit_ms;                     /* host wall time of the last call spent describing the batch and enqueueing work */
    float host_wait_ms;                       /* host wall time of the last call spent waiting for the device */
    int32_t devices;                          /* GPUs the last call was sharded over (ROCJPEG_B200_DEVICES) */
    uint64_t entries;                         /* 32-bit coefficient entries the entropy stage wrote (pad entries included) */
    uint32_t truncated_images;                /* pictures of the last call whose scan ended before their last block */
    uint32_t pad_;
    uint64_t fused_blocks;                    /* blocks transformed by the fused IDCT + output kernel (whole-picture RGB / RGB_PLANAR):
                                                 their planes never reach memory */
} RocJpegB200Stats;

/* CUDA-event timing on a decoder handle: 0 off (default), 1 an event after every stage (stage_ms and total_ms;
 * the events keep neighbouring stages from overlapping), 2 first and last event only (total_ms).
 * Env ROCJPEG_B200_PROFILE sets the initial level. */
RocJpegStatus rocJpegB200SetProfiling(RocJpegHandle handle, int enable);
/* Colour convention of RGB and RGB_PLANAR outputs, per handle. It applies to every later rocJpegDecode,
 * rocJpegDecodeBatched, rocJpegB200DecodeBatchedScaled and rocJpegB200Prepare[Scaled] on the handle (and to the other
 * devices of a sharded call); rocJpegB200Run replays what Prepare captured.
 *   ROCJPEG_B200_COLOR_REFERENCE (default): the reference's kernels, BT.709 full-range float and nearest-neighbour chroma;
 *   ROCJPEG_B200_COLOR_LIBJPEG: libjpeg-turbo's default decode (what Pillow and torchvision's CPU decoder return), JFIF
 *     integer colour and "fancy" (triangle) chroma upsampling, bit for bit at full size and at 1/2, 1/4, 1/8 except for
 *     4:2:0 at a reduced size (libjpeg-turbo transforms that chroma at twice the luma size instead of upsampling it).
 * NATIVE, YUV_PLANAR and Y outputs, and 4:0:0 pictures, are the same under both. An unknown value returns
 * ROCJPEG_STATUS_INVALID_PARAMETER. Env ROCJPEG_B200_COLOR=libjpeg sets the initial convention at rocJpegCreate. */
#define ROCJPEG_B200_COLOR_REFERENCE 0
#define ROCJPEG_B200_COLOR_LIBJPEG 1
RocJpegStatus rocJpegB200SetColorConvention(RocJpegHandle handle, int convention);
RocJpegStatus rocJpegB200GetColorConvention(RocJpegHandle handle, int *convention);
/* Statistics of the last rocJpegDecode / rocJpegDecodeBatched / rocJpegB200Run on this handle. */
RocJpegStatus rocJpegB200GetStats(RocJpegHandle handle, RocJpegB200Stats *stats);

/* Split form of rocJpegDecodeBatched: Prepare parses nothing new — it builds the batch description
 * and copies descriptors + entropy-coded bytes to the device; Run launches every stage on the
 * resident batch and synchronises. Run may be called repeatedly. */
RocJpegStatus rocJpegB200Prepare(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles, int batch_size,
                                 const RocJpegDecodeParams *decode_params, RocJpegImage *destinations);
RocJpegStatus rocJpegB200Run(RocJpegHandle handle);

/* Decode at reduced size. Denominator d in {1, 2, 4, 8} per picture: the picture is decoded with libjpeg's reduced
 * inverse DCTs (jidctred.c; an 8x8 block becomes an (8/d)x(8/d) block), so the entropy decode is the same and the
 * transform and everything after it do 1/d^2 of the work. The output is ceil(W/d) x ceil(H/d) luma samples (libjpeg's
 * output_width / output_height for scale_num 1, scale_denom d); every RocJpegImage layout rule of rocJpegDecodeBatched
 * applies to that size, and the crop rectangle is given in its coordinates. Every component is transformed at the same
 * reduced size, so chroma keeps its coded ratio (libjpeg-turbo decodes 4:2:0 chroma with the next larger transform
 * instead, to save upsampling; the results of the two differ in 4:2:0 chroma only). d = 1 is rocJpegDecodeBatched
 * itself. A denominator outside {1, 2, 4, 8} returns ROCJPEG_STATUS_INVALID_PARAMETER. RocJpegDecodeParams'
 * target_dimension keeps the meaning it has for rocJpegDecodeBatched (none).
 *   rocJpegB200GetScaledImageInfo: the sizes a decode at 1/scale_denom writes (the rocJpegGetImageInfo rules applied to
 *     ceil(W/d) x ceil(H/d));
 *   rocJpegB200DecodeBatchedScaled: rocJpegDecodeBatched with one denominator per picture (scale_denoms NULL: all 1);
 *   rocJpegB200PrepareScaled: rocJpegB200Prepare with denominators; rocJpegB200Run is unchanged.
 * After a scaled decode rocJpegB200GetPlanes returns the scaled planes: component c is (blocks_w[c] * 8/d) x
 * (blocks_h[c] * 8/d) samples; rocJpegB200GetCoefficients is unchanged. */
RocJpegStatus rocJpegB200GetScaledImageInfo(RocJpegHandle handle, RocJpegStreamHandle jpeg_stream_handle, int scale_denom, uint8_t *num_components,
                                            RocJpegChromaSubsampling *subsampling, uint32_t *widths, uint32_t *heights);
RocJpegStatus rocJpegB200DecodeBatchedScaled(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles, int batch_size,
                                             const RocJpegDecodeParams *decode_params, const int32_t *scale_denoms, RocJpegImage *destinations);
RocJpegStatus rocJpegB200PrepareScaled(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles, int batch_size,
                                       const RocJpegDecodeParams *decode_params, const int32_t *scale_denoms, RocJpegImage *destinations);

/* Decode straight to a requested size, resampled as Pillow does (Image.resize), on the GPU behind the decode. Per picture:
 *   1. decode exactly as rocJpegB200DecodeBatchedScaled would: the handle's colour convention, at 1/scale_denom, the crop
 *      rectangle of decode_params in the scaled picture's coordinates;
 *   2. resize that picture to width x height with Pillow's Image.resize((width, height), filter), byte for byte: Pillow's
 *      double-precision weights rounded to 22-bit fixed point, a horizontal then a vertical pass of int32 multiply-adds with
 *      the clipped 8-bit intermediate in between (Pillow's Resample.c).
 * With a crop the result is img.crop(box).resize(size, filter): torchvision's resized_crop on a PIL image.
 * Output formats at the requested size: RGB (interleaved, channel[0]), RGB_PLANAR (three planes, all with pitch[0]), Y
 * (luma only: Pillow's "L" mode). Any pitch of at least the row's bytes, any base alignment. NATIVE and YUV_PLANAR,
 * filter 0 (NEAREST) or any other unknown filter, a width or height of 0 or above 65535, a denominator outside
 * {1, 2, 4, 8}, a null channel or a pitch below the row's bytes return ROCJPEG_STATUS_INVALID_PARAMETER before anything
 * runs. Per-image status, BAD_JPEG and ROCJPEG_B200_STRICT behave as for rocJpegDecodeBatched; a truncated picture is
 * resized from what its decode produced. The decoded pictures pass through a device arena the handle keeps (grow-only).
 * A resized call runs on the handle's own device: on a sharded handle (ROCJPEG_B200_DEVICES) it is not split, and a
 * destination on another device returns ROCJPEG_STATUS_INVALID_PARAMETER. target_dimension stays unread.
 *   rocJpegB200DecodeBatchedResized: resize[i] for picture i;
 *   rocJpegB200PrepareResized: rocJpegB200Prepare with resizes; rocJpegB200Run replays it unchanged;
 *   rocJpegB200ResizeCoefficients (host only): Pillow's coefficients of one axis, as the passes apply them.
 *     *ksize = taps per output sample (2 ceil(support) + 1); bounds[2 i] = first input sample of output sample i,
 *     bounds[2 i + 1] = how many it reads; taps[i * ksize + t] = their fixed-point weights, rows padded with zeros.
 *     bounds and taps NULL: only *ksize. capacity (in taps) below out_size * ksize: INVALID_PARAMETER. */
#define ROCJPEG_B200_FILTER_LANCZOS 1 /* Pillow's Image.Resampling values */
#define ROCJPEG_B200_FILTER_BILINEAR 2
#define ROCJPEG_B200_FILTER_BICUBIC 3
#define ROCJPEG_B200_FILTER_BOX 4
#define ROCJPEG_B200_FILTER_HAMMING 5
typedef struct {
    uint32_t width, height; /* size of the output, >= 1 each */
    int32_t filter;         /* ROCJPEG_B200_FILTER_* */
    int32_t scale_denom;    /* 1, 2, 4, 8: reduced-size IDCT before the resize (as rocJpegB200DecodeBatchedScaled) */
} RocJpegB200Resize;
RocJpegStatus rocJpegB200DecodeBatchedResized(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles, int batch_size,
                                              const RocJpegDecodeParams *decode_params, const RocJpegB200Resize *resize,
                                              RocJpegImage *destinations);
RocJpegStatus rocJpegB200PrepareResized(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles, int batch_size,
                                        const RocJpegDecodeParams *decode_params, const RocJpegB200Resize *resize,
                                        RocJpegImage *destinations);
RocJpegStatus rocJpegB200ResizeCoefficients(uint32_t in_size, uint32_t out_size, int filter, int32_t *bounds, int32_t *taps,
                                            size_t capacity, int32_t *ksize);

/* Timing-harness helper: exactly the caller's loop of the reference's batched sample - rocJpegStreamParse(datas[i],
 * lengths[i], handles[i]) for every image, then one rocJpegDecodeBatched - issued from C. *parse_seconds (optional) = wall
 * time of the parse loop. */
RocJpegStatus rocJpegB200ParseAndDecodeBatched(RocJpegHandle handle, RocJpegStreamHandle *jpeg_stream_handles,
                                               const unsigned char *const *datas, const size_t *lengths, int batch_size,
                                               const RocJpegDecodeParams *decode_params, RocJpegImage *destinations,
                                               double *parse_seconds);

/* File -> device ingestion (opt-in; the callers' I/O in the reference's samples is one ifstream read per image into a
 * pageable vector on the decode thread, samples/rocjpeg_samples_utils.h:213-234 and
 * samples/jpegDecodeBatched/jpegdecodebatched.cpp:106-121): `io_threads` threads (<= 0: 8) read paths[i] straight into
 * stream handle i's pooled page-locked staging and parse it there, equivalent to rocJpegStreamParse on the file's bytes
 * but without the intermediate copy - rocJpegDecodeBatched then uploads from that memory in place. per_file_status
 * (optional) receives one status per file: SUCCESS, INVALID_PARAMETER (cannot open / read), BAD_JPEG. Returns the first
 * failure, or SUCCESS. */
RocJpegStatus rocJpegB200StreamLoadFiles(RocJpegStreamHandle *jpeg_stream_handles, const char *const *paths, int count,
                                         int io_threads, RocJpegStatus *per_file_status);

/* Stage taps for image `index` of the last decoded batch. Layout = the oracle's: component-major,
 * each component an MCU-padded raster of blocks (64 int16, natural order) / samples (u8; at scale 1/d
 * (8/d)x(8/d) samples per block, see rocJpegB200DecodeBatchedScaled). */
RocJpegStatus rocJpegB200GetCoefficients(RocJpegHandle handle, int index, int16_t *host_out, size_t count);
RocJpegStatus rocJpegB200GetPlanes(RocJpegHandle handle, int index, uint8_t *host_out, size_t count);

/* Taps on the GPU destuffing pass (k0_destuff.cu) for image `index` of the last decoded batch: what it found in the
 * raw bytes, and the destuffed bytes of one restart interval as they lie in device memory. */
typedef struct {
    uint32_t segments_seen;  /* restart intervals present in the bytes (restart markers + 1) */
    uint32_t scan_size;      /* raw bytes up to the first FF D9 - what the reference's parser computes on the host
                                (src/rocjpeg_parser.cpp:400-416) */
    uint32_t flags;          /* ROCJPEG_B200_SCAN_* */
    uint32_t reserved;
} RocJpegB200ScanStatus;
#define ROCJPEG_B200_SCAN_NO_EOI 1u            /* no FF D9: the slice ran to the end of the buffer */
#define ROCJPEG_B200_SCAN_STRAY_MARKER 2u      /* a marker other than RSTn / EOI inside the entropy-coded data */
#define ROCJPEG_B200_SCAN_EXTRA_RESTARTS 4u    /* more restart markers than the frame has restart intervals */
#define ROCJPEG_B200_SCAN_MISSING_INTERVALS 8u /* fewer restart intervals in the bytes than the frame needs */
#define ROCJPEG_B200_SCAN_EMPTY_INTERVAL 16u   /* a restart interval that must hold blocks holds no bytes */
#define ROCJPEG_B200_DECODE_SHORT 32u          /* a restart interval ran out of bytes before its last block */
#define ROCJPEG_B200_TRUNCATED_MASK (8u | 16u | 32u)
RocJpegStatus rocJpegB200GetScanStatus(RocJpegHandle handle, int index, RocJpegB200ScanStatus *status);
/* Per-image outcome of the last rocJpegDecode / rocJpegDecodeBatched: ROCJPEG_B200_SCAN_* | ROCJPEG_B200_DECODE_* flags.
 * Every picture of a batch is decoded as far as its bytes go (blocks a truncated or damaged scan does not reach are
 * zero: mid grey). When any picture has a ROCJPEG_B200_TRUNCATED_MASK flag the decode call returns
 * ROCJPEG_STATUS_BAD_JPEG (the reference's VCN path reports a failed surface as an error too,
 * src/rocjpeg_vaapi_decoder.cpp:846-868, and stops its batch there); this tells which pictures and why. Environment
 * ROCJPEG_B200_STRICT=0 keeps the return code at SUCCESS. */
RocJpegStatus rocJpegB200GetImageStatus(RocJpegHandle handle, int index, uint32_t *flags);
RocJpegStatus rocJpegB200GetDeviceSegment(RocJpegHandle handle, int index, uint32_t segment, uint8_t *host_out, size_t capacity,
                                          uint32_t *nbytes);

/* Parser taps (host only). */
typedef struct {
    int32_t width, height, num_components, chroma_subsampling;
    int32_t h_sampling[3], v_sampling[3], quant_selector[3], dc_selector[3], ac_selector[3];
    int32_t restart_interval;
    uint32_t num_mcus;                /* as the reference computes it (src/rocjpeg_parser.cpp:197) */
    uint32_t scan_offset;             /* first entropy-coded byte inside the caller's buffer */
    uint32_t raw_bytes;               /* from there to the end of the buffer (the slice ends at the first FF D9: found on the GPU) */
    int32_t mcus_x, mcus_y, blocks_per_mcu;
    int32_t blocks_w[3], blocks_h[3];
    uint32_t num_segments;            /* restart intervals the frame needs, bounded by what the bytes can hold */
    int32_t decode_status;            /* RocJpegStatus rocJpegDecode would return for this stream */
    int32_t source_is_device_visible; /* the entropy-coded bytes are in page-locked memory (the caller's or the staging pool's) */
    int32_t source_is_zero_copy;      /* ... the caller's own page-locked buffer, used in place */
    int32_t features;                 /* ROCJPEG_B200_FEAT_*: what the stream uses beyond what the reference's parser accepts */
} RocJpegB200StreamInfo;
/* Accepted here, rejected by the reference's parser (SURVEY.md section 8 f4): an SOF1 frame header with 8-bit samples (the
 * sequential Huffman process is the same decode; libjpeg-turbo writes SOF1 as soon as a quantiser step exceeds 255),
 * quantiser tables with 16-bit steps (src/rocjpeg_parser.cpp:230) and Huffman table ids 2 and 3 (:274). */
#define ROCJPEG_B200_FEAT_SOF1 1
#define ROCJPEG_B200_FEAT_DQT16 2
#define ROCJPEG_B200_FEAT_HUFF_ID23 4
RocJpegStatus rocJpegB200StreamGetInfo(RocJpegStreamHandle jpeg_stream_handle, RocJpegB200StreamInfo *info);
/* The HOST restatement of the GPU destuffing pass (tests and taps only - rocJpegStreamParse does not touch the
 * entropy-coded bytes and the decode path never runs this): slice size up to the first FF D9 as the reference's
 * parser reports it (src/rocjpeg_parser.cpp:400-416), restart markers, destuffed restart intervals. Reads the
 * caller's buffer given to the last rocJpegStreamParse, which must still be valid. */
typedef struct {
    uint32_t scan_size;
    uint32_t restart_markers_seen;
    uint32_t num_segments;
    uint64_t clean_bytes;             /* destuffed stream incl. per-segment padding */
} RocJpegB200HostScanInfo;
RocJpegStatus rocJpegB200StreamHostScan(RocJpegStreamHandle jpeg_stream_handle, RocJpegB200HostScanInfo *info);
/* Copy the destuffed bytes of restart interval `segment` as the host restatement produces them (returns its
 * length via *nbytes). */
RocJpegStatus rocJpegB200StreamGetSegment(RocJpegStreamHandle jpeg_stream_handle, uint32_t segment, uint8_t *out,
                                          size_t capacity, uint32_t *nbytes);
/* Why the last rocJpegStreamParse on this handle failed (the text the library also prints to stderr, as the
 * reference does through ERR - src/rocjpeg_commons.h); empty after a successful parse. NUL-terminated, truncated
 * to `capacity`. */
RocJpegStatus rocJpegB200StreamGetLastError(RocJpegStreamHandle jpeg_stream_handle, char *out, size_t capacity);
/* Tables as the decoder sees them: quantiser steps in natural order; Huffman BITS/HUFFVAL. */
RocJpegStatus rocJpegB200StreamGetQuantTable(RocJpegStreamHandle jpeg_stream_handle, int id, uint16_t out_natural[64]);
RocJpegStatus rocJpegB200StreamGetHuffmanTable(RocJpegStreamHandle jpeg_stream_handle, int is_ac, int id, uint8_t bits[16],
                                               uint8_t vals[256], uint32_t *count);

/* Multi-GPU sharding of rocJpegDecodeBatched (images are independent: no collective). With the environment variable
 * ROCJPEG_B200_DEVICES=N (N > 1) set when rocJpegCreate runs, the handle also drives the N-1 devices after device_id.
 * Each batch is then split over the devices: an image whose destination buffer lives on one of those peer devices is
 * decoded there (nothing of it crosses a link); the others - destinations on the handle's own device, the layout of the
 * reference's samples - are dealt by the longest-processing-time rule on entropy-coded bytes, and the shares of the
 * peers are delivered into the handle's device over NVLink (row-wise stores of the output stage through peer access).
 * Every device decodes its share concurrently; the join is one stream sync per device. A destination on a device the
 * handle does not drive is rejected (INVALID_PARAMETER).
 * rocJpegB200PlanShards / ...Pinned expose the assignment rule (host only): cost[i] = entropy-coded bytes of image i,
 * fixed[i] >= 0 pins image i to that device (fixed may be NULL), out_device[i] in [0, num_devices) = index among the
 * devices the handle drives (0 = device_id). rocJpegB200GetDeviceCount = devices the handle drives. */
RocJpegStatus rocJpegB200PlanShards(const uint64_t *cost, int batch_size, int num_devices, int *out_device);
RocJpegStatus rocJpegB200PlanShardsPinned(const uint64_t *cost, const int *fixed, int batch_size, int num_devices, int *out_device);
RocJpegStatus rocJpegB200GetDeviceCount(RocJpegHandle handle, int *num_devices);

const char *rocJpegB200Version(void);

#if defined(__cplusplus)
}
#endif
#endif /* ROCJPEG_B200_EXT_H */
