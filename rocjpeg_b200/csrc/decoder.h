// decoder.h — host orchestrator of the CUDA decode pipeline.
//
// Counterpart of the reference's RocJpegDecoder (src/rocjpeg_decoder.h:45-176,
// src/rocjpeg_decoder.cpp) with its VA-API back end (RocJpegVappiDecoder,
// src/rocjpeg_vaapi_decoder.h:274-413) folded in: where the reference submits
// one picture at a time to a VCN core, waits on the surface, imports it into HIP
// and launches a post-processing kernel per image, this class describes a whole
// batch in one descriptor block, uploads it with the entropy-coded bytes, and
// runs one launch per stage (K1 sync rounds, K1 write, DC scan, K2, K3) over all
// images on the handle's CUDA stream. Device arenas are grow-only and reused
// across calls (the reference's surface pool, vaapi_decoder.h:113-215).
#pragma once
#include <cuda_runtime_api.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "device_types.h"
#include "jpeg_parser.h"
#include "resample.h"
#include "stages.h"

namespace rjb {

// Mirrors RocJpegDecodeParams / RocJpegImage (include/rocjpeg.h) without
// depending on the public header.
struct DecodeParams {
    int32_t output_format;
    int16_t crop_left, crop_top, crop_right, crop_bottom;
    int32_t color = 0;   // kColor*: the handle's colour convention (not part of RocJpegDecodeParams)
};
// Colour conventions of RGB / RGB_PLANAR (ROCJPEG_B200_COLOR_* of include/rocjpeg_b200_ext.h)
constexpr int kColorReference = 0;   // the reference's kernels: BT.709 full-range float, nearest-neighbour chroma
constexpr int kColorLibjpeg = 1;     // libjpeg-turbo's default decode: JFIF integer colour, fancy upsampling (k3_jfif.cu)
struct DestImage {
    uint8_t* channel[4];
    uint32_t pitch[4];
    int32_t scale_denom;   // 1, 2, 4 or 8: the picture is decoded at 1/scale_denom of its size (reduced-size IDCT)
};
constexpr int kScaledKernels = 3;   // reduced-size IDCT kernels: scale 1/2, 1/4, 1/8
inline bool ValidScale(int d) { return d == 1 || d == 2 || d == 4 || d == 8; }
inline int ScaleIndex(int d) { return d == 2 ? 0 : d == 4 ? 1 : 2; }   // d > 1: index of its reduced-size kernel
// Size and filter of one picture of a resized decode (RocJpegB200Resize without the denominator, which DestImage carries)
struct ResizeSpec {
    uint32_t width, height;   // 1 .. kMaxResizeSize
    int32_t filter;           // ResampleFilter (resample.h)
};

// The argument checks of a resized decode that need no device: formats (RGB, RGB_PLANAR, Y), filters, sizes, denominators,
// destination channels and pitches. nullptr when they hold, else why not (INVALID_PARAMETER).
const char* CheckResizeArgs(const DecodeParams& params, int n, const DestImage* dsts, const ResizeSpec* resize);

class DeviceBuffer {
  public:
    DeviceBuffer() = default;
    ~DeviceBuffer();
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    cudaError_t Reserve(size_t bytes);   // grow-only; contents lost on growth
    template <class U> U* as() const { return reinterpret_cast<U*>(ptr_); }
    size_t capacity() const { return cap_; }

  private:
    void* ptr_ = nullptr;
    size_t cap_ = 0;
};

enum StageId {
    kStageUpload = 0,   // descriptor block + entropy-coded bytes, host -> device
    kStageDestuff,      // K0: end of slice, destuffing, restart intervals, segment table (three launches)
    kStageSync,         // all k1_sync rounds
    kStageWrite,        // k1_scan + k1_write
    kStageDc,           // dc_sums + dc_scan + dc_apply (none when k1_fused integrates the DC)
    kStageIdct,         // k2_idct and the reduced-size k2_idct_4x4 / 2x2 / 1x1
    kStageOutput,       // k3_output
    kStageCount
};

struct BatchStats {
    float stage_ms[kStageCount] = {};
    float total_ms = 0;                 // first event to last event
    uint32_t sync_rounds = 0;           // k1_sync launches that were needed
    uint32_t decodes_per_round[kMaxSyncRounds] = {};
    uint64_t scan_bytes = 0;            // entropy-coded bytes as uploaded
    uint64_t blocks = 0;                // 8x8 blocks decoded
    uint64_t entries = 0;               // 32-bit coefficient entries K1 wrote (pad entries included)
    uint64_t subsequences = 0;
    uint64_t plane_bytes = 0;           // bytes of decoded component planes (K2 output)
    uint64_t fused_blocks = 0;          // blocks the fused IDCT + output kernel transformed (their planes never reach memory)
    uint64_t output_bytes = 0;          // bytes K3 writes
    uint64_t h2d_bytes = 0, d2h_bytes = 0;
    uint32_t kernel_launches = 0;
    int sub_bytes = 0;
    int lanes = 0;                      // pipeline lanes (chunks) the batch was split over
    float host_submit_ms = 0, host_wait_ms = 0;   // host wall time: describing + enqueueing / waiting for the device
    int devices = 1;                    // GPUs the call was sharded over
    uint32_t truncated_images = 0;      // pictures whose scan ended before their last block
    // adds another lane's or device's counters: sums, and the larger sync_rounds and sub_bytes (not total_ms, lanes,
    // devices, truncated_images, host_*_ms)
    void Accumulate(const BatchStats& s);
};

// Helper threads of one decoder: they copy pageable input into page-locked staging, and a sharded call enqueues
// each device's share from one of them. Workers sleep on a condition variable between calls.
class SubmitPool {
  public:
    explicit SubmitPool(int workers);
    ~SubmitPool();
    SubmitPool(const SubmitPool&) = delete;
    SubmitPool& operator=(const SubmitPool&) = delete;
    // fn(0) on the calling thread, fn(1..n-1) on the workers; returns when all are done
    void Run(int n, const std::function<void(int)>& fn);

  private:
    void Loop(int index);
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_;
    uint64_t generation_ = 0;
    int jobs_ = 0;
    const std::function<void(int)>* fn_ = nullptr;
    std::atomic<int> pending_{0};
    bool stop_ = false;
};

// One pipeline lane: a CUDA stream, its device arenas and the description of the
// (sub-)batch it is decoding. A decode call splits its batch over up to kMaxLanes lanes so
// that the upload of one chunk overlaps the kernels of another and the latency-bound tails
// of the entropy stage overlap across chunks.
class Lane {
  public:
    Lane() = default;
    ~Lane();
    Lane(const Lane&) = delete;
    Lane& operator=(const Lane&) = delete;
    int Create(int device_id, int sm_count, bool prealloc = true);
    // remote[i] != 0: image i's destination lives on another GPU (stores go over NVLink: rows through the output stage, not the
    // IDCT stage's scattered block stores); nullptr: all local
    // resize != nullptr (one per picture): the pictures are decoded into the lane's resize arena and resized from there into
    // dsts (RGB_PLANAR is decoded interleaved, the vertical pass writes the planes)
    int Build(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const uint8_t* remote = nullptr,
              const ResizeSpec* resize = nullptr);
    int Upload(cudaStream_t upload_stream);   // nullptr: use the lane's own stream
    int LaunchAll(bool include_upload, int profiling, cudaStream_t upload_stream);
    int Finish(int profiling);
    int Sync();
    int WaitEvent(cudaEvent_t ev);   // the lane's later work waits for `ev`
    int CopyCoefficients(int image, int16_t* host_out, size_t count);
    int CopyPlanes(int image, uint8_t* host_out, size_t count);
    int CopySegment(int image, uint32_t segment, uint8_t* host_out, size_t capacity, uint32_t* nbytes);
    int GetScanStatus(int image, ScanStatus* out) const;
    const BatchStats& stats() const { return stats_; }
    const std::string& last_error() const { return err_; }
    cudaEvent_t first_event() const { return ev_[0]; }
    cudaEvent_t last_event() const { return ev_[kStageCount]; }
    int num_images() const { return int(h_images_.size()); }
    uint32_t truncated_images() const { return truncated_images_; }
    // ROCJPEG_B200_TRACE=2: one line per lane, device times relative to `origin` (the first lane's upload-begin event)
    void PrintTimeline(int index, cudaEvent_t origin, double host_origin_ms) const;
    cudaEvent_t trace_origin() const { return ev_trace_[0]; }
    void set_host_mark(int i, double ms) { host_ms_[i] = ms; }

  private:
    struct Layout;   // byte layout of the descriptor block
    int Fail(int status, const std::string& why);
    // the IDCT stage: k2_idct for the full-size pictures, a reduced-size kernel per scale present; counts the launches
    int LaunchIdct(bool force_planes, uint32_t* launches);
    // Everything after the entropy stage: DC integration (integrate_dc), IDCT, fused IDCT + output, output stage, then
    // the counters and per-image status back to the host. mark(i) runs after stage i - 1 (LaunchAll's stage events).
    int LaunchDownstream(bool integrate_dc, const std::function<cudaError_t(int)>& mark);
    // the resize jobs and tables of a resized call, the arena they live in, and the decode's destinations inside it
    int PlanResize(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const ResizeSpec* resize);

    bool created_ = false;
    std::string err_;
    cudaStream_t stream_ = nullptr;
    cudaEvent_t ev_[kStageCount + 1] = {};
    cudaEvent_t ev_uploaded_ = nullptr;
    cudaEvent_t ev_trace_[3] = {};   // ROCJPEG_B200_TRACE=2: upload begins / upload done / last kernel done, on the device's clock
    double host_ms_[3] = {};         // ... and when the host began describing the lane, began enqueueing, was done with it
    int sm_count_ = 0;

    // host-side batch description
    std::vector<ImageDesc> h_images_;
    std::vector<OutputDesc> h_outputs_;
    std::vector<uint32_t> h_img_cta0_, h_img_dctile0_, h_k2_tile0_, h_k3_tile0_, h_k0_tile0_, h_needed_segments_;
    std::vector<uint32_t> h_k2s_tile0_[kScaledKernels];   // first tile of each image in the reduced-size kernel of its scale
    std::vector<int> h_scale_;                             // scale denominator of each image
    uint32_t truncated_images_ = 0;
    std::vector<GatherItem> h_gather_;
    struct CopyRun {
        const uint8_t* src;   // host address (page-locked), 16-byte aligned
        uint64_t dst_off;     // offset in the raw arena
        size_t nbytes;
    };
    std::vector<CopyRun> h_runs_;          // upload plan: neighbouring streams of one page-locked allocation move with one copy
    std::vector<FusedImage> h_fused_;      // pictures served by the fused IDCT + output kernel
    std::vector<uint32_t> h_tile_img_;     // per strip of the strip kernel (k23_fused): index into h_fused_
    std::vector<uint32_t> h_tile_img_w_;   // ... of the warp-per-column kernel (k23_warp: aligned destinations)
    std::vector<const HuffLutSet*> h_lut_ptrs_;
    std::vector<const ParsedJpeg*> h_lut_specs_;
    std::vector<uint64_t> h_lut_hashes_;
    std::vector<uint16_t> h_qtables_;
    K0Args k0_ = {};
    K1Args k1_ = {};
    K2Args k2_ = {};
    K2Args k2s_[kScaledKernels] = {};   // reduced-size IDCT: the pictures of scale 1/2, 1/4, 1/8
    K3Args k3_ = {};
    K23Args k23_ = {};
    K4Args k4_ = {};
    std::vector<ResizeJob> h_resize_;          // resized calls: one job per picture (empty otherwise)
    std::vector<int32_t> h_resize_coef_;       // their tables (K4Args::coef)
    std::vector<uint32_t> h_rh_tile0_, h_rv_tile0_;
    std::vector<DestImage> h_resize_dsts_;     // where the decode writes each picture: the resize arena
    DeviceBuffer d_resize_;                    // decoded pictures + intermediate rows (grow-only)
    bool jfif_ = false;           // the output stage is k3_jfif (RGB / RGB_PLANAR under the libjpeg colour convention)
    bool k2_needed_ = true;       // some image of the lane is not served by the fused kernel
    bool any_direct_ = false, needs_planes_ = false;
    // The kernel schedule, fixed by Build: how the entropy-coded bytes are uploaded (the gather kernel also leaves the
    // destuffing pass's per-tile prefix elements), and k1_fused or `sync_rounds_` k1_sync rounds up front + k1_write.
    enum UploadBy { kUploadPerPicture, kUploadRuns, kUploadGather } upload_by_ = kUploadPerPicture;
    bool k1_fused_ = false;
    bool inline_destuff_ = false;   // k1_fused destuffs the raw bytes itself, no K0 runs (chosen by Build, replayed by every Run)
    bool clean_valid_ = false;      // the clean stream and the segment table hold the current batch (K0 ran)
    int sync_rounds_ = 2;
    size_t scan_bytes_ = 0, raw_bytes_ = 0, coef_blocks_ = 0, entry_count_ = 0, plane_bytes_ = 0, nsub_total_ = 0;
    uint32_t nseg_total_ = 0;

    StagingBuffer h_desc_;        // pinned descriptor block
    size_t desc_bytes_ = 0;
    StagingBuffer h_counters_;    // pinned read-back
    DeviceBuffer d_slab_;         // descriptors, scan bytes, K1 state, coefficient entries, block records: one allocation
    DeviceBuffer d_planes_;       // component planes, only when some image needs the output stage
    DeviceBuffer d_counters_;     // two sets of K1 counters: a batch uses one, its write pass zeroes the other for the next
    int counter_set_ = 0;
    BatchStats stats_;
};

constexpr int kMaxLanes = 8;      // lanes a handle owns; how many a call uses: Decoder::Split
constexpr int kMaxDevices = 16;



// Longest-processing-time-first assignment of `n` independent images (cost = entropy-coded bytes)
// to `ndev` devices: images in decreasing cost order, each to the least loaded device. Images are
// independent units (no exchange step, SURVEY.md section 8e), so this is the whole "parallelism
// plan" of a sharded rocJpegDecodeBatched. out_device[i] in [0, ndev).
void PlanShards(const uint64_t* cost, int n, int ndev, int* out_device);
// The same with some images already placed: fixed[i] >= 0 pins image i to that device (its destination buffer lives
// there), fixed[i] < 0 leaves it to the rule; the pinned images' costs count as load before the others are dealt.
void PlanShardsPinned(const uint64_t* cost, const int* fixed, int n, int ndev, int* out_device);

class Decoder {
  public:
    Decoder(int backend, int device_id);
    ~Decoder();
    int Initialize();   // RocJpegStatus
    // scale_denom > 1: the sizes a decode at that scale writes (rocJpegB200GetScaledImageInfo)
    int GetImageInfo(const StreamParser* s, uint8_t* ncomp, int32_t* css, uint32_t* widths, uint32_t* heights, int scale_denom = 1);
    // resize != nullptr: rocJpegB200DecodeBatchedResized (one spec per picture; never sharded: the handle's own device)
    int Decode(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const ResizeSpec* resize = nullptr);

    // Extension entry points (include/rocjpeg_b200_ext.h)
    int Prepare(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const ResizeSpec* resize = nullptr);
    int Run();          // launch all stages for the prepared batch and synchronise
    int CopyCoefficients(int image, int16_t* host_out, size_t count);   // component-major raster layout
    int CopyPlanes(int image, uint8_t* host_out, size_t count);
    int CopySegment(int image, uint32_t segment, uint8_t* host_out, size_t capacity, uint32_t* nbytes);   // destuffed by K0
    int GetScanStatus(int image, ScanStatus* out);
    void SetProfiling(int level) { profiling_ = level; }   // 0 off, 1 per-stage events, 2 first/last event only
    // kColor*: applies to every later decode and Prepare on this handle, the peers of a sharded call included
    void SetColorConvention(int convention);
    int color_convention() const { return color_; }
    const BatchStats& stats() const { return stats_; }
    const std::string& last_error() const { return err_; }
    int device_id() const { return device_id_; }
    int num_devices() const { return 1 + int(peers_.size()); }

  private:
    // Sharded form of Decode: the batch is split over this handle's device and its peers
    // (ROCJPEG_B200_DEVICES), every device runs the whole pipeline on its share concurrently and
    // writes its pixels straight into the caller's buffers (peer stores over NVLink when the
    // buffer lives on another GPU). No collective: the join is one stream sync per device.
    int DecodeSharded(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts);
    int Submit(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const uint8_t* remote);   // async part
    int Wait();
    int RecordCaller();   // ev_caller_ on this device's legacy default stream, behind what the caller enqueued there so far
    int Fail(int status, const std::string& why);
    int Split(const StreamParser* const* streams, int n);
    int BuildAll(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, bool launch, const uint8_t* remote = nullptr,
                 const ResizeSpec* resize = nullptr);
    // the device check of a call that is not sharded (one picture, a resized call, Prepare): on a sharded handle every
    // destination must live on this handle's own device - the call writes from that device only, after the caller's work
    // on that device's legacy default stream only
    int CheckOwnDevice(int n, const DecodeParams& params, const DestImage* dsts);
    int FinishAll();
    void Aggregate();
    // image index of the last call -> the decoder (this or a peer) and lane that holds it, index inside the lane
    Lane* Locate(int image, int* local);

    int backend_, device_id_;
    bool initialized_ = false, prepared_ = false;
    bool strict_status_ = true;   // ROCJPEG_B200_STRICT=0: truncated scans do not change the return code
    int profiling_ = 0;
    int color_ = kColorReference;
    std::mutex mutex_;
    std::string err_;
    int sm_count_ = 0;
    Lane lanes_[kMaxLanes];
    cudaStream_t upload_stream_ = nullptr;   // all host->device traffic, serialised in lane order
    // Recorded on the device's legacy default stream at the start of a call that writes the caller's memory; the call's
    // work waits for it. The lanes' and the upload stream are non-blocking, so without it a decode would overwrite a
    // destination that work the caller has already enqueued there (a framework's default stream) still writes or reads.
    cudaEvent_t ev_caller_ = nullptr;
    int active_lanes_ = 0;
    int chunk_first_[kMaxLanes + 1] = {};   // image range of each lane's chunk
    BatchStats stats_;
    // multi-device sharding
    std::unique_ptr<SubmitPool> pool_;              // copiers of pageable input into staging (ROCJPEG_B200_COPY_THREADS)
    std::unique_ptr<SubmitPool> shard_pool_;        // one submitter per peer device
    bool is_peer_ = false;                          // a peer never shards further
    std::vector<std::unique_ptr<Decoder>> peers_;   // decoders on the other devices, owned by the handle's decoder
    std::vector<int> shard_dev_, shard_local_;      // image -> (0 = this device, k = peers_[k-1]; index inside that device's share)
    bool sharded_ = false;
};

}  // namespace rjb
