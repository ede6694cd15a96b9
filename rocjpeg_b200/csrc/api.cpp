// api.cpp — the C ABI of librocjpeg.so.
//
// Same nine entry points, argument checks and status codes as the reference's
// src/rocjpeg_api.cpp (null arguments -> INVALID_PARAMETER :39,69,87,108,133,162,
// 195,223; parse failure -> BAD_JPEG :73-75; C++ exception -> RUNTIME_ERROR
// :170-174; handle allocation failure -> NOT_INITIALIZED :45-48,113-116; error
// names :246-277), over this repository's parser and CUDA decoder. Handle
// wrappers mirror src/rocjpeg_api_decoder_handle.h / rocjpeg_api_stream_handle.h
// (object + last-error string). The rocJpegB200* extension entry points are
// declared in include/rocjpeg_b200_ext.h.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <cstring>
#include <exception>
#include <iostream>
#include <memory>
#include <string>
#include <vector>

#include "decoder.h"
#include "jpeg_parser.h"
#include "rocjpeg_b200_ext.h"

#define ERR(X) std::cerr << "[ERR] " << " {" << __func__ << "} " << " " << X << std::endl;

namespace {

struct StreamHandle {
    std::shared_ptr<rjb::StreamParser> parser = std::make_shared<rjb::StreamParser>();
    std::string error;
};

struct DecoderHandle {
    DecoderHandle(RocJpegBackend backend, int device_id) : decoder(std::make_shared<rjb::Decoder>(int(backend), device_id)) {}
    std::shared_ptr<rjb::Decoder> decoder;
    std::string error;
    void CaptureError(const std::string& m) { error = m; }
};

inline rjb::DecodeParams ToParams(const RocJpegDecodeParams* p) {
    rjb::DecodeParams d;
    d.output_format = int32_t(p->output_format);
    d.crop_left = p->crop_rectangle.left;
    d.crop_top = p->crop_rectangle.top;
    d.crop_right = p->crop_rectangle.right;
    d.crop_bottom = p->crop_rectangle.bottom;
    return d;
}

// The decoder's destinations: the caller's RocJpegImage plus the picture's scale denominator (scale_denoms NULL: all 1).
// INVALID_PARAMETER for a denominator other than 1, 2, 4 or 8.
int ToDests(const RocJpegImage* images, int n, const int32_t* scale_denoms, std::vector<rjb::DestImage>* out) {
    out->resize(size_t(n));
    for (int i = 0; i < n; i++) {
        rjb::DestImage& d = (*out)[size_t(i)];
        for (int c = 0; c < 4; c++) {
            d.channel[c] = images[i].channel[c];
            d.pitch[c] = images[i].pitch[c];
        }
        d.scale_denom = scale_denoms ? scale_denoms[i] : 1;
        if (!rjb::ValidScale(d.scale_denom)) return ROCJPEG_STATUS_INVALID_PARAMETER;
    }
    return ROCJPEG_STATUS_SUCCESS;
}
static_assert(ROCJPEG_B200_STAGE_COUNT == rjb::kStageCount, "stage count");

int CollectStreams(RocJpegStreamHandle* handles, int n, std::vector<const rjb::StreamParser*>* out) {
    out->resize(size_t(n));
    for (int i = 0; i < n; i++) {
        if (handles[i] == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
        (*out)[size_t(i)] = static_cast<StreamHandle*>(handles[i])->parser.get();
    }
    return ROCJPEG_STATUS_SUCCESS;
}

}  // namespace

extern "C" {

RocJpegStatus ROCJPEGAPI rocJpegStreamCreate(RocJpegStreamHandle* jpeg_stream_handle) {
    if (jpeg_stream_handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    StreamHandle* h = nullptr;
    try {
        h = new StreamHandle();
    } catch (const std::exception& e) {
        ERR(std::string("Failed to init the rocJPEG stream handle, ") + e.what());
        return ROCJPEG_STATUS_NOT_INITIALIZED;
    }
    *jpeg_stream_handle = h;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus ROCJPEGAPI rocJpegStreamParse(const unsigned char* data, size_t length, RocJpegStreamHandle jpeg_stream_handle) {
    if (data == nullptr || jpeg_stream_handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<StreamHandle*>(jpeg_stream_handle);
    try {
        if (!h->parser->Parse(data, length)) {
            h->error = h->parser->last_error();
            ERR("Invalid JPEG! " + h->error);
            return ROCJPEG_STATUS_BAD_JPEG;
        }
        h->error.clear();
    } catch (const std::exception& e) {
        h->error = e.what();
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus ROCJPEGAPI rocJpegStreamDestroy(RocJpegStreamHandle jpeg_stream_handle) {
    if (jpeg_stream_handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    delete static_cast<StreamHandle*>(jpeg_stream_handle);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus ROCJPEGAPI rocJpegCreate(RocJpegBackend backend, int device_id, RocJpegHandle* handle) {
    if (handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    DecoderHandle* h = nullptr;
    try {
        h = new DecoderHandle(backend, device_id);
    } catch (const std::exception& e) {
        ERR(std::string("Failed to init the rocJPEG handle, ") + e.what());
        return ROCJPEG_STATUS_NOT_INITIALIZED;
    }
    // as in the reference (src/rocjpeg_api.cpp:118-119) the handle is handed out before
    // initialisation runs: a failed init still leaves the caller a handle to destroy
    *handle = h;
    try {
        RocJpegStatus st = RocJpegStatus(h->decoder->Initialize());
        if (st != ROCJPEG_STATUS_SUCCESS) h->CaptureError(h->decoder->last_error());
        return st;
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

RocJpegStatus ROCJPEGAPI rocJpegDestroy(RocJpegHandle handle) {
    if (handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    delete static_cast<DecoderHandle*>(handle);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus ROCJPEGAPI rocJpegGetImageInfo(RocJpegHandle handle, RocJpegStreamHandle jpeg_stream_handle, uint8_t* num_components,
                                             RocJpegChromaSubsampling* subsampling, uint32_t* widths, uint32_t* heights) {
    if (handle == nullptr || num_components == nullptr || subsampling == nullptr || widths == nullptr || heights == nullptr)
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    if (jpeg_stream_handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;   // src/rocjpeg_decoder.cpp:309-311
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        int32_t css = 0;
        int st = h->decoder->GetImageInfo(static_cast<StreamHandle*>(jpeg_stream_handle)->parser.get(), num_components, &css, widths, heights);
        *subsampling = RocJpegChromaSubsampling(css);
        return RocJpegStatus(st);
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

RocJpegStatus rocJpegB200GetScaledImageInfo(RocJpegHandle handle, RocJpegStreamHandle jpeg_stream_handle, int scale_denom, uint8_t* num_components,
                                            RocJpegChromaSubsampling* subsampling, uint32_t* widths, uint32_t* heights) {
    if (handle == nullptr || jpeg_stream_handle == nullptr || num_components == nullptr || subsampling == nullptr || widths == nullptr ||
        heights == nullptr || !rjb::ValidScale(scale_denom))
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        int32_t css = 0;
        int st = h->decoder->GetImageInfo(static_cast<StreamHandle*>(jpeg_stream_handle)->parser.get(), num_components, &css, widths, heights,
                                          scale_denom);
        *subsampling = RocJpegChromaSubsampling(css);
        return RocJpegStatus(st);
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

RocJpegStatus ROCJPEGAPI rocJpegDecode(RocJpegHandle handle, RocJpegStreamHandle jpeg_stream_handle, const RocJpegDecodeParams* decode_params,
                                       RocJpegImage* destination) {
    if (handle == nullptr || decode_params == nullptr || destination == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    if (jpeg_stream_handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;   // src/rocjpeg_decoder.cpp:107-109
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        const rjb::StreamParser* s = static_cast<StreamHandle*>(jpeg_stream_handle)->parser.get();
        std::vector<rjb::DestImage> dsts;
        ToDests(destination, 1, nullptr, &dsts);
        int st = h->decoder->Decode(&s, 1, ToParams(decode_params), dsts.data());
        if (st != 0) h->CaptureError(h->decoder->last_error());
        return RocJpegStatus(st);
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

RocJpegStatus ROCJPEGAPI rocJpegDecodeBatched(RocJpegHandle handle, RocJpegStreamHandle* jpeg_stream_handles, int batch_size,
                                              const RocJpegDecodeParams* decode_params, RocJpegImage* destinations) {
    return rocJpegB200DecodeBatchedScaled(handle, jpeg_stream_handles, batch_size, decode_params, nullptr, destinations);
}

RocJpegStatus rocJpegB200DecodeBatchedScaled(RocJpegHandle handle, RocJpegStreamHandle* jpeg_stream_handles, int batch_size,
                                             const RocJpegDecodeParams* decode_params, const int32_t* scale_denoms, RocJpegImage* destinations) {
    if (handle == nullptr || jpeg_stream_handles == nullptr || decode_params == nullptr || destinations == nullptr)
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        if (batch_size < 0) return ROCJPEG_STATUS_INVALID_PARAMETER;
        std::vector<const rjb::StreamParser*> streams;
        int st = CollectStreams(jpeg_stream_handles, batch_size, &streams);
        if (st != 0) return RocJpegStatus(st);
        std::vector<rjb::DestImage> dsts;
        st = ToDests(destinations, batch_size, scale_denoms, &dsts);
        if (st != 0) return RocJpegStatus(st);
        st = h->decoder->Decode(streams.data(), batch_size, ToParams(decode_params), dsts.data());
        if (st != 0) h->CaptureError(h->decoder->last_error());
        return RocJpegStatus(st);
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

// src/rocjpeg_api.cpp:246-277
const char* ROCJPEGAPI rocJpegGetErrorName(RocJpegStatus rocjpeg_status) {
    switch (rocjpeg_status) {
        case ROCJPEG_STATUS_SUCCESS: return "ROCJPEG_STATUS_SUCCESS";
        case ROCJPEG_STATUS_NOT_INITIALIZED: return "ROCJPEG_STATUS_NOT_INITIALIZED";
        case ROCJPEG_STATUS_INVALID_PARAMETER: return "ROCJPEG_STATUS_INVALID_PARAMETER";
        case ROCJPEG_STATUS_BAD_JPEG: return "ROCJPEG_STATUS_BAD_JPEG";
        case ROCJPEG_STATUS_JPEG_NOT_SUPPORTED: return "ROCJPEG_STATUS_JPEG_NOT_SUPPORTED";
        case ROCJPEG_STATUS_EXECUTION_FAILED: return "ROCJPEG_STATUS_EXECUTION_FAILED";
        case ROCJPEG_STATUS_ARCH_MISMATCH: return "ROCJPEG_STATUS_ARCH_MISMATCH";
        case ROCJPEG_STATUS_INTERNAL_ERROR: return "ROCJPEG_STATUS_INTERNAL_ERROR";
        case ROCJPEG_STATUS_IMPLEMENTATION_NOT_SUPPORTED: return "ROCJPEG_STATUS_IMPLEMENTATION_NOT_SUPPORTED";
        case ROCJPEG_STATUS_HW_JPEG_DECODER_NOT_SUPPORTED: return "ROCJPEG_STATUS_HW_JPEG_DECODER_NOT_SUPPORTED";
        case ROCJPEG_STATUS_RUNTIME_ERROR: return "ROCJPEG_STATUS_RUNTIME_ERROR";
        case ROCJPEG_STATUS_OUTOF_MEMORY: return "ROCJPEG_STATUS_OUTOF_MEMORY";
        case ROCJPEG_STATUS_NOT_IMPLEMENTED: return "ROCJPEG_STATUS_NOT_IMPLEMENTED";
        default: return "UNKNOWN_ERROR";
    }
}

// ------------------------------------------------------------------ extensions

RocJpegStatus rocJpegB200SetProfiling(RocJpegHandle handle, int enable) {
    if (handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    static_cast<DecoderHandle*>(handle)->decoder->SetProfiling(enable);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200GetStats(RocJpegHandle handle, RocJpegB200Stats* stats) {
    if (handle == nullptr || stats == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    const rjb::BatchStats& s = static_cast<DecoderHandle*>(handle)->decoder->stats();
    std::memset(stats, 0, sizeof(*stats));
    for (int i = 0; i < ROCJPEG_B200_STAGE_COUNT; i++) stats->stage_ms[i] = s.stage_ms[i];
    stats->total_ms = s.total_ms;
    stats->sync_rounds = s.sync_rounds;
    for (int i = 0; i < 8; i++) stats->decodes_per_round[i] = s.decodes_per_round[i];
    stats->scan_bytes = s.scan_bytes;
    stats->blocks = s.blocks;
    stats->subsequences = s.subsequences;
    stats->plane_bytes = s.plane_bytes;
    stats->output_bytes = s.output_bytes;
    stats->h2d_bytes = s.h2d_bytes;
    stats->d2h_bytes = s.d2h_bytes;
    stats->kernel_launches = s.kernel_launches;
    stats->subsequence_bytes = s.sub_bytes;
    stats->lanes = s.lanes;
    stats->host_submit_ms = s.host_submit_ms;
    stats->host_wait_ms = s.host_wait_ms;
    stats->devices = s.devices;
    stats->entries = s.entries;
    stats->truncated_images = s.truncated_images;
    stats->fused_blocks = s.fused_blocks;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200Prepare(RocJpegHandle handle, RocJpegStreamHandle* jpeg_stream_handles, int batch_size,
                                 const RocJpegDecodeParams* decode_params, RocJpegImage* destinations) {
    return rocJpegB200PrepareScaled(handle, jpeg_stream_handles, batch_size, decode_params, nullptr, destinations);
}

RocJpegStatus rocJpegB200PrepareScaled(RocJpegHandle handle, RocJpegStreamHandle* jpeg_stream_handles, int batch_size,
                                       const RocJpegDecodeParams* decode_params, const int32_t* scale_denoms, RocJpegImage* destinations) {
    if (handle == nullptr || jpeg_stream_handles == nullptr || decode_params == nullptr || destinations == nullptr || batch_size <= 0)
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        std::vector<const rjb::StreamParser*> streams;
        int st = CollectStreams(jpeg_stream_handles, batch_size, &streams);
        if (st != 0) return RocJpegStatus(st);
        std::vector<rjb::DestImage> dsts;
        st = ToDests(destinations, batch_size, scale_denoms, &dsts);
        if (st != 0) return RocJpegStatus(st);
        return RocJpegStatus(h->decoder->Prepare(streams.data(), batch_size, ToParams(decode_params), dsts.data()));
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

RocJpegStatus rocJpegB200Run(RocJpegHandle handle) {
    if (handle == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<DecoderHandle*>(handle);
    try {
        return RocJpegStatus(h->decoder->Run());
    } catch (const std::exception& e) {
        h->CaptureError(e.what());
        ERR(e.what());
        return ROCJPEG_STATUS_RUNTIME_ERROR;
    }
}

// The caller's loop of the reference's batched sample (samples/jpegDecodeBatched/jpegdecodebatched.cpp:106-160):
// rocJpegStreamParse per image, then one rocJpegDecodeBatched - the public entry points, called from C so that
// a timing harness written in Python measures the library and not its own interpreter.
RocJpegStatus rocJpegB200ParseAndDecodeBatched(RocJpegHandle handle, RocJpegStreamHandle* jpeg_stream_handles, const unsigned char* const* datas,
                                               const size_t* lengths, int batch_size, const RocJpegDecodeParams* decode_params,
                                               RocJpegImage* destinations, double* parse_seconds) {
    if (handle == nullptr || jpeg_stream_handles == nullptr || datas == nullptr || lengths == nullptr || batch_size < 0)
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < batch_size; i++) {
        const RocJpegStatus st = rocJpegStreamParse(datas[i], lengths[i], jpeg_stream_handles[i]);
        if (st != ROCJPEG_STATUS_SUCCESS) return st;
    }
    if (parse_seconds) *parse_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return rocJpegDecodeBatched(handle, jpeg_stream_handles, batch_size, decode_params, destinations);
}

// File -> device ingestion: `io_threads` threads read the files straight into the stream handles' pooled page-locked
// staging and parse them there (rjb::StreamParser::ParseFile).
RocJpegStatus rocJpegB200StreamLoadFiles(RocJpegStreamHandle* jpeg_stream_handles, const char* const* paths, int count, int io_threads,
                                         RocJpegStatus* per_file_status) {
    if (jpeg_stream_handles == nullptr || paths == nullptr || count < 0) return ROCJPEG_STATUS_INVALID_PARAMETER;
    for (int i = 0; i < count; i++)
        if (jpeg_stream_handles[i] == nullptr || paths[i] == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    const int nthreads = std::max(1, std::min(io_threads <= 0 ? 8 : io_threads, std::max(count, 1)));
    std::vector<RocJpegStatus> status(size_t(count), ROCJPEG_STATUS_SUCCESS);
    std::atomic<int> next{0};
    auto work = [&]() {
        for (;;) {
            const int i = next.fetch_add(1, std::memory_order_relaxed);
            if (i >= count) return;
            auto h = static_cast<StreamHandle*>(jpeg_stream_handles[i]);
            try {
                const int rc = h->parser->ParseFile(paths[i]);
                h->error = rc == 0 ? std::string() : h->parser->last_error();
                status[size_t(i)] = rc == 0 ? ROCJPEG_STATUS_SUCCESS : rc == -2 ? ROCJPEG_STATUS_INVALID_PARAMETER : ROCJPEG_STATUS_BAD_JPEG;
            } catch (const std::exception& e) {
                h->error = e.what();
                status[size_t(i)] = ROCJPEG_STATUS_RUNTIME_ERROR;
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; t++) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    RocJpegStatus first = ROCJPEG_STATUS_SUCCESS;
    for (int i = 0; i < count; i++) {
        if (per_file_status) per_file_status[i] = status[size_t(i)];
        if (status[size_t(i)] != ROCJPEG_STATUS_SUCCESS && first == ROCJPEG_STATUS_SUCCESS) first = status[size_t(i)];
    }
    return first;
}

RocJpegStatus rocJpegB200PlanShards(const uint64_t* cost, int batch_size, int num_devices, int* out_device) {
    if (cost == nullptr || out_device == nullptr || batch_size < 0 || num_devices < 1) return ROCJPEG_STATUS_INVALID_PARAMETER;
    rjb::PlanShards(cost, batch_size, num_devices, out_device);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200PlanShardsPinned(const uint64_t* cost, const int* fixed, int batch_size, int num_devices, int* out_device) {
    if (cost == nullptr || out_device == nullptr || batch_size < 0 || num_devices < 1) return ROCJPEG_STATUS_INVALID_PARAMETER;
    rjb::PlanShardsPinned(cost, fixed, batch_size, num_devices, out_device);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200GetDeviceCount(RocJpegHandle handle, int* num_devices) {
    if (handle == nullptr || num_devices == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    *num_devices = static_cast<DecoderHandle*>(handle)->decoder->num_devices();
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200GetCoefficients(RocJpegHandle handle, int index, int16_t* host_out, size_t count) {
    if (handle == nullptr || host_out == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    return RocJpegStatus(static_cast<DecoderHandle*>(handle)->decoder->CopyCoefficients(index, host_out, count));
}

RocJpegStatus rocJpegB200GetPlanes(RocJpegHandle handle, int index, uint8_t* host_out, size_t count) {
    if (handle == nullptr || host_out == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    return RocJpegStatus(static_cast<DecoderHandle*>(handle)->decoder->CopyPlanes(index, host_out, count));
}

RocJpegStatus rocJpegB200GetDeviceSegment(RocJpegHandle handle, int index, uint32_t segment, uint8_t* host_out, size_t capacity, uint32_t* nbytes) {
    if (handle == nullptr || nbytes == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    return RocJpegStatus(static_cast<DecoderHandle*>(handle)->decoder->CopySegment(index, segment, host_out, capacity, nbytes));
}

RocJpegStatus rocJpegB200GetScanStatus(RocJpegHandle handle, int index, RocJpegB200ScanStatus* status) {
    if (handle == nullptr || status == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    rjb::ScanStatus st;
    const int rc = static_cast<DecoderHandle*>(handle)->decoder->GetScanStatus(index, &st);
    if (rc != 0) return RocJpegStatus(rc);
    status->segments_seen = st.segments_seen;
    status->scan_size = st.scan_size;
    status->flags = st.flags;
    status->reserved = st.reserved;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200GetImageStatus(RocJpegHandle handle, int index, uint32_t* flags) {
    if (handle == nullptr || flags == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    rjb::ScanStatus st;
    const int rc = static_cast<DecoderHandle*>(handle)->decoder->GetScanStatus(index, &st);
    if (rc != 0) return RocJpegStatus(rc);
    *flags = st.flags;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamGetInfo(RocJpegStreamHandle jpeg_stream_handle, RocJpegB200StreamInfo* info) {
    if (jpeg_stream_handle == nullptr || info == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<StreamHandle*>(jpeg_stream_handle);
    const rjb::ParsedJpeg& p = h->parser->parsed();
    std::memset(info, 0, sizeof(*info));
    if (!p.valid) return ROCJPEG_STATUS_BAD_JPEG;
    info->width = p.width; info->height = p.height; info->num_components = p.ncomp; info->chroma_subsampling = p.css;
    for (int c = 0; c < 3; c++) {
        info->h_sampling[c] = p.hs[c]; info->v_sampling[c] = p.vs[c]; info->quant_selector[c] = p.tq[c];
        info->dc_selector[c] = p.td[c]; info->ac_selector[c] = p.ta[c];
        info->blocks_w[c] = p.blocks_w[c]; info->blocks_h[c] = p.blocks_h[c];
    }
    info->restart_interval = p.restart_interval;
    info->num_mcus = p.num_mcus_ref;
    info->scan_offset = p.scan_offset;
    info->raw_bytes = p.raw_bytes;
    info->mcus_x = p.mcus_x; info->mcus_y = p.mcus_y; info->blocks_per_mcu = p.bpm;
    info->num_segments = p.nseg;
    info->decode_status = p.support_status;
    info->source_is_device_visible = h->parser->raw().dev != nullptr ? 1 : 0;
    info->source_is_zero_copy = h->parser->raw().zero_copy ? 1 : 0;
    info->features = p.features;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamGetSegment(RocJpegStreamHandle jpeg_stream_handle, uint32_t segment, uint8_t* out, size_t capacity,
                                          uint32_t* nbytes) {
    if (jpeg_stream_handle == nullptr || nbytes == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<StreamHandle*>(jpeg_stream_handle);
    const rjb::ParsedJpeg& p = h->parser->parsed();
    if (!p.valid) return ROCJPEG_STATUS_BAD_JPEG;
    const rjb::HostScan& hs = h->parser->host_scan();
    if (!hs.done || segment >= hs.segments.size()) return ROCJPEG_STATUS_INVALID_PARAMETER;
    const rjb::Segment& s = hs.segments[segment];
    *nbytes = s.nbytes;
    if (out != nullptr) {
        if (capacity < s.nbytes) return ROCJPEG_STATUS_INVALID_PARAMETER;
        std::memcpy(out, hs.clean.data() + s.offset, s.nbytes);
    }
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamHostScan(RocJpegStreamHandle jpeg_stream_handle, RocJpegB200HostScanInfo* info) {
    if (jpeg_stream_handle == nullptr || info == nullptr) return ROCJPEG_STATUS_INVALID_PARAMETER;
    auto h = static_cast<StreamHandle*>(jpeg_stream_handle);
    if (!h->parser->parsed().valid) return ROCJPEG_STATUS_BAD_JPEG;
    const rjb::HostScan& hs = h->parser->host_scan();
    if (!hs.done) return ROCJPEG_STATUS_INVALID_PARAMETER;
    info->scan_size = hs.scan_size;
    info->restart_markers_seen = hs.restart_markers_seen;
    info->num_segments = uint32_t(hs.segments.size());
    info->clean_bytes = hs.clean_bytes;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamGetLastError(RocJpegStreamHandle jpeg_stream_handle, char* out, size_t capacity) {
    if (jpeg_stream_handle == nullptr || out == nullptr || capacity == 0) return ROCJPEG_STATUS_INVALID_PARAMETER;
    const std::string& e = static_cast<StreamHandle*>(jpeg_stream_handle)->error;
    const size_t n = std::min(e.size(), capacity - 1);
    std::memcpy(out, e.data(), n);
    out[n] = 0;
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamGetQuantTable(RocJpegStreamHandle jpeg_stream_handle, int id, uint16_t out_natural[64]) {
    if (jpeg_stream_handle == nullptr || out_natural == nullptr || id < 0 || id >= 4) return ROCJPEG_STATUS_INVALID_PARAMETER;
    const rjb::ParsedJpeg& p = static_cast<StreamHandle*>(jpeg_stream_handle)->parser->parsed();
    if (!p.valid || !p.qt_present[id]) return ROCJPEG_STATUS_BAD_JPEG;
    std::memcpy(out_natural, p.qt_natural[id], 128);
    return ROCJPEG_STATUS_SUCCESS;
}

RocJpegStatus rocJpegB200StreamGetHuffmanTable(RocJpegStreamHandle jpeg_stream_handle, int is_ac, int id, uint8_t bits[16],
                                               uint8_t vals[256], uint32_t* count) {
    if (jpeg_stream_handle == nullptr || bits == nullptr || vals == nullptr || count == nullptr || id < 0 || id >= rjb::kHuffIds)
        return ROCJPEG_STATUS_INVALID_PARAMETER;
    const rjb::ParsedJpeg& p = static_cast<StreamHandle*>(jpeg_stream_handle)->parser->parsed();
    if (!p.valid) return ROCJPEG_STATUS_BAD_JPEG;
    const rjb::HuffSpec& t = is_ac ? p.ac[id] : p.dc[id];
    if (!t.present) return ROCJPEG_STATUS_BAD_JPEG;
    std::memcpy(bits, t.bits, 16);
    std::memcpy(vals, t.vals, 256);
    *count = t.count;
    return ROCJPEG_STATUS_SUCCESS;
}

const char* rocJpegB200Version(void) { return "rocjpeg-b200 0.6.0 (sm_100a)"; }

}  // extern "C"
