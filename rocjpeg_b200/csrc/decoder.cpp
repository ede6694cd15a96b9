// decoder.cpp — see decoder.h. Status codes are RocJpegStatus values
// (include/rocjpeg.h); error behaviour follows src/rocjpeg_decoder.cpp and
// src/rocjpeg_commons.h:43-65 of the reference (print to stderr, return a code).
#include "decoder.h"

#include "huff_core.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>

namespace rjb {

namespace {
constexpr int kSuccess = 0, kNotInitialized = -1, kInvalidParameter = -2, kBadJpeg = -3, kNotSupported = -4,
              kOutOfMemory = -5, kExecutionFailed = -6, kNotImplemented = -12;

inline size_t AlignUp(size_t v, size_t a) { return (v + a - 1) / a * a; }

int EnvInt(const char* name, int dflt) {
    const char* v = std::getenv(name);
    return (v && *v) ? std::atoi(v) : dflt;
}

int TraceLevel() {
    static const int level = EnvInt("ROCJPEG_B200_TRACE", 0);
    return level;
}

double NowMs() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        if (changed) cudaSetDevice(prev);
    }
};

#define RJB_CUDA(call)                                                                                       \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess) {                                                                             \
            std::cerr << "CUDA failure: 'status: " << cudaGetErrorName(e_) << "' at " << __FILE__ << ":" << __LINE__ \
                      << std::endl;                                                                          \
            return Fail(e_ == cudaErrorMemoryAllocation ? kOutOfMemory : kExecutionFailed, cudaGetErrorString(e_)); \
        }                                                                                                    \
    } while (0)
}  // namespace

SubmitPool::SubmitPool(int workers) {
    for (int i = 0; i < workers; i++) threads_.emplace_back([this, i] { Loop(i + 1); });
}

SubmitPool::~SubmitPool() {
    {
        std::lock_guard<std::mutex> lock(m_);
        stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
}

void SubmitPool::Loop(int index) {
    uint64_t seen = 0;
    for (;;) {
        const std::function<void(int)>* fn = nullptr;
        {
            std::unique_lock<std::mutex> lock(m_);
            cv_.wait(lock, [&] { return stop_ || generation_ != seen; });
            if (stop_) return;
            seen = generation_;
            if (index < jobs_) fn = fn_;
        }
        if (fn) {
            (*fn)(index);
            pending_.fetch_sub(1, std::memory_order_acq_rel);
        }
    }
}

void SubmitPool::Run(int n, const std::function<void(int)>& fn) {
    n = std::min(n, int(threads_.size()) + 1);
    {
        std::lock_guard<std::mutex> lock(m_);
        fn_ = &fn;
        jobs_ = n;
        pending_.store(n - 1, std::memory_order_release);
        generation_++;
    }
    cv_.notify_all();
    fn(0);
    while (pending_.load(std::memory_order_acquire) != 0) std::this_thread::yield();
}

namespace {
// Waits for the submitter's turn on the shared upload stream and passes it on - also when the
// submitter bails out early, so that the lanes behind it never wait forever.
struct TurnGuard {
    UploadTurn t;
    bool passed = false;
    explicit TurnGuard(UploadTurn turn) : t(turn) {}
    void Acquire() const {
        if (t.turn)
            while (t.turn->load(std::memory_order_acquire) != t.mine) std::this_thread::yield();
    }
    void Release() {
        if (t.turn && !passed) t.turn->store(t.mine + 1, std::memory_order_release);
        passed = true;
    }
    ~TurnGuard() {
        if (!passed) {
            Acquire();
            Release();
        }
    }
};
}  // namespace

DeviceBuffer::~DeviceBuffer() {
    if (ptr_) cudaFree(ptr_);
}

cudaError_t DeviceBuffer::Reserve(size_t bytes) {
    if (bytes <= cap_) return cudaSuccess;
    if (ptr_) {
        cudaError_t e = cudaFree(ptr_);
        ptr_ = nullptr;
        cap_ = 0;
        if (e != cudaSuccess) return e;
    }
    size_t want = AlignUp(bytes + bytes / 8, 1 << 20);
    cudaError_t e = cudaMalloc(&ptr_, want);
    if (e != cudaSuccess) {
        ptr_ = nullptr;
        return e;
    }
    cap_ = want;
    return cudaSuccess;
}

Lane::~Lane() {
    if (!created_) return;
    for (auto& e : ev_)
        if (e) cudaEventDestroy(e);
    if (ev_uploaded_) cudaEventDestroy(ev_uploaded_);
    for (auto& e : ev_trace_)
        if (e) cudaEventDestroy(e);
    if (stream_) cudaStreamDestroy(stream_);
}

int Lane::Fail(int status, const std::string& why) {
    err_ = why;
    return status;
}

int Lane::Create(int /*device_id*/, int sm_count, bool prealloc) {
    if (created_) return kSuccess;
    sm_count_ = sm_count;
    RJB_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    for (auto& ev : ev_) RJB_CUDA(cudaEventCreate(&ev));
    RJB_CUDA(cudaEventCreateWithFlags(&ev_uploaded_, cudaEventDisableTiming));
    if (TraceLevel() >= 2)
        for (auto& ev : ev_trace_) RJB_CUDA(cudaEventCreate(&ev));
    // what a first call would otherwise allocate inside its timed region (the reference's perf sample
    // times every call, the first included; a cold cudaMalloc was measured at 1-26 ms): page-locked
    // staging and a starting size for the device arenas, ROCJPEG_B200_PREALLOC_MB per handle (default
    // 384, two thirds of it arena, one third planes, split over the lanes; 0 = allocate on demand)
    if (!h_desc_.Reserve(1u << 20) || !h_counters_.Reserve(256 + 4096 * sizeof(ScanStatus))) return Fail(kOutOfMemory, "page-locked staging");
    const size_t per_lane = size_t(std::max(0, EnvInt("ROCJPEG_B200_PREALLOC_MB", 384))) * (1u << 20) / 4;   // (the lanes a call uses by default)
    RJB_CUDA(d_counters_.Reserve(512));
    RJB_CUDA(cudaMemsetAsync(d_counters_.as<uint8_t>(), 0, 512, stream_));
    if (per_lane && prealloc) {
        RJB_CUDA(d_slab_.Reserve(per_lane * 2 / 3));
        RJB_CUDA(d_planes_.Reserve(per_lane / 3));
    }
    created_ = true;
    return kSuccess;
}

int Lane::Sync() {
    RJB_CUDA(cudaStreamSynchronize(stream_));
    return kSuccess;
}

Decoder::Decoder(int backend, int device_id) : backend_(backend), device_id_(device_id) {}

Decoder::~Decoder() {   // lanes release their own streams, events and arenas
    if (upload_stream_) cudaStreamDestroy(upload_stream_);
}

int Decoder::Fail(int status, const std::string& why) {
    err_ = why;
    return status;
}

// src/rocjpeg_decoder.cpp:46-91 (InitHIP + InitializeDecoder)
int Decoder::Initialize() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1) {
        (void)cudaGetLastError();
        std::cerr << "[ERR]  {Initialize}  ERROR: Failed to find any GPU!" << std::endl;
        return Fail(kNotInitialized, "no CUDA device");
    }
    if (device_id_ < 0 || device_id_ >= count) {
        std::cerr << "[ERR]  {Initialize}  ERROR: the requested device_id is not found!" << std::endl;
        return Fail(kInvalidParameter, "device_id out of range");
    }
    if (backend_ == 1) return Fail(kNotImplemented, "ROCJPEG_BACKEND_HYBRID is not implemented");   // decoder.cpp:87-88
    if (backend_ != 0) return Fail(kInvalidParameter, "unknown backend");
    DeviceGuard guard(device_id_);
    RJB_CUDA(cudaSetDevice(device_id_));
    cudaDeviceProp prop;
    RJB_CUDA(cudaGetDeviceProperties(&prop, device_id_));
    sm_count_ = prop.multiProcessorCount;
    int st = lanes_[0].Create(device_id_, sm_count_);
    if (st != kSuccess) return Fail(st, lanes_[0].last_error());
    // the upload stream outranks the lanes' streams: the CTAs of the gather kernel (PCIe-bound, few) must
    // not queue behind the thousands of CTAs of another lane's decode kernels
    int prio_lo = 0, prio_hi = 0;
    RJB_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    RJB_CUDA(cudaStreamCreateWithPriority(&upload_stream_, cudaStreamNonBlocking, prio_hi));
    profiling_ = EnvInt("ROCJPEG_B200_PROFILE", 0);
    strict_status_ = EnvInt("ROCJPEG_B200_STRICT", 1) != 0;
    // everything a first decode would otherwise pay for: kernel modules, the lanes' streams and events
    RJB_CUDA(PreloadK0());
    RJB_CUDA(PreloadK1());
    RJB_CUDA(PreloadK2());
    RJB_CUDA(PreloadK2Scaled());
    RJB_CUDA(PreloadK3());
    RJB_CUDA(PreloadK23());
    for (int l = 1; l < 4; l++) {   // the lanes a call uses by default; the others (ROCJPEG_B200_LANES > 4) are created on demand
        st = lanes_[l].Create(device_id_, sm_count_);
        if (st != kSuccess) return Fail(st, lanes_[l].last_error());
    }
    initialized_ = true;
    // Multi-device sharding of rocJpegDecodeBatched (the C API has no way to ask for it, hence the
    // environment variable): peers = the next devices after device_id, each reachable with peer
    // access so that its output stage can store into buffers on this handle's device.
    const int want = is_peer_ ? 1 : std::min(EnvInt("ROCJPEG_B200_DEVICES", 1), std::min(count, kMaxDevices));
    for (int k = 1; k < want; k++) {
        const int dev = (device_id_ + k) % count;
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dev, device_id_) != cudaSuccess || !can) {
            (void)cudaGetLastError();
            std::cerr << "[WARN] rocjpeg_b200: device " << dev << " cannot access device " << device_id_ << " memory; not used for sharding" << std::endl;
            continue;
        }
        std::unique_ptr<Decoder> peer(new Decoder(backend_, dev));
        peer->is_peer_ = true;
        if (peer->Initialize() != kSuccess) continue;
        {
            DeviceGuard pg(dev);
            cudaError_t pe = cudaDeviceEnablePeerAccess(device_id_, 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) {
                (void)cudaGetLastError();
                continue;
            }
            (void)cudaGetLastError();
        }
        peer->profiling_ = profiling_;
        peers_.push_back(std::move(peer));
    }
    return kSuccess;
}

namespace {
// Device that owns a device pointer; -1 for anything else (host memory, null, unknown). *base / *size (optional) = the
// allocation the pointer lies in: destinations carved from one allocation (a framework's caching allocator) cost one
// driver query, not one per picture.
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

int DeviceOfPointer(const void* p, uintptr_t* base = nullptr, size_t* size = nullptr) {
    if (base) *base = 0;
    if (size) *size = 0;
    if (!p) return -1;
    if (PointerAttributesFn fn = DriverPointerAttributes()) {
        // CU_POINTER_ATTRIBUTE_MEMORY_TYPE = 2, DEVICE_ORDINAL = 9, RANGE_START_ADDR = 11, RANGE_SIZE = 12
        int which[4] = {2, 9, 11, 12};
        unsigned int mem_type = 0;
        int ordinal = -1;
        unsigned long long start = 0;
        size_t bytes = 0;
        void* out[4] = {&mem_type, &ordinal, &start, &bytes};
        if (fn(4, which, out, static_cast<unsigned long long>(reinterpret_cast<uintptr_t>(p))) == 0) {
            if (mem_type != 2u /* CU_MEMORYTYPE_DEVICE */) return -1;
            if (base) *base = uintptr_t(start);
            if (size) *size = bytes;
            return ordinal;
        }
    }
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return -1;
    }
    return at.type == cudaMemoryTypeDevice ? at.device : -1;
}
}  // namespace

void PlanShards(const uint64_t* cost, int n, int ndev, int* out_device) { PlanShardsPinned(cost, nullptr, n, ndev, out_device); }

void PlanShardsPinned(const uint64_t* cost, const int* fixed, int n, int ndev, int* out_device) {
    if (ndev < 1) ndev = 1;
    std::vector<int> order;
    order.reserve(size_t(std::max(n, 0)));
    std::vector<uint64_t> load(size_t(ndev), 0);
    for (int i = 0; i < n; i++) {
        if (fixed && fixed[i] >= 0 && fixed[i] < ndev) {
            out_device[i] = fixed[i];
            load[size_t(fixed[i])] += cost[i] + 1;
        } else {
            order.push_back(i);
        }
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    for (int i : order) {
        int best = 0;
        for (int d = 1; d < ndev; d++)
            if (load[size_t(d)] < load[size_t(best)]) best = d;
        out_device[i] = best;
        load[size_t(best)] += cost[i] + 1;   // +1: zero-cost images still spread out
    }
}

// src/rocjpeg_decoder.cpp:307-358
int Decoder::GetImageInfo(const StreamParser* s, uint8_t* ncomp, int32_t* css, uint32_t* widths, uint32_t* heights, int scale_denom) {
    std::lock_guard<std::mutex> lock(mutex_);
    if (!s || !ncomp || !css || !widths || !heights || !ValidScale(scale_denom)) return kInvalidParameter;
    const ParsedJpeg& p = s->parsed();
    *ncomp = uint8_t(p.ncomp);
    *css = p.css;
    // at scale 1/d the picture is ceil(W/d) x ceil(H/d) (libjpeg's output_width / output_height), the rules below apply to that
    widths[0] = uint32_t((p.width + scale_denom - 1) / scale_denom);
    heights[0] = uint32_t((p.height + scale_denom - 1) / scale_denom);
    widths[3] = heights[3] = 0;
    switch (p.css) {
        case CSS_444: widths[1] = widths[2] = widths[0]; heights[1] = heights[2] = heights[0]; break;
        case CSS_440: widths[1] = widths[2] = widths[0]; heights[1] = heights[2] = heights[0] >> 1; break;
        case CSS_422: widths[1] = widths[2] = widths[0] >> 1; heights[1] = heights[2] = heights[0]; break;
        case CSS_420: widths[1] = widths[2] = widths[0] >> 1; heights[1] = heights[2] = heights[0] >> 1; break;
        case CSS_400: widths[1] = widths[2] = 0; heights[1] = heights[2] = 0; break;
        case CSS_411: widths[1] = widths[2] = widths[0] >> 2; heights[1] = heights[2] = heights[0]; break;
        default: break;
    }
    return kSuccess;
}

// Bytes the output stage writes for one image (valid bytes only), mirroring the
// sizing rules of samples/rocjpeg_samples_utils.h:318-399.
static uint64_t OutputBytes(int css, int fmt, int W, int H) {
    const int sx = css == CSS_411 ? 2 : (css == CSS_422 || css == CSS_420) ? 1 : 0, sy = (css == CSS_440 || css == CSS_420) ? 1 : 0;
    const uint64_t luma = uint64_t(W) * H;
    switch (fmt) {
        case FMT_RGB:
        case FMT_RGB_PLANAR: return 3 * luma;
        case FMT_Y: return luma;
        case FMT_YUV_PLANAR: return css == CSS_400 ? luma : luma + 2ull * uint64_t(W >> sx) * uint64_t(H >> sy);
        case FMT_NATIVE:
            if (css == CSS_400) return luma;
            if (css == CSS_422) return 2 * luma;
            if (css == CSS_420) return luma + uint64_t(W) * uint64_t(H >> 1);
            return luma + 2ull * uint64_t(W >> sx) * uint64_t(H >> sy);
        default: return 0;
    }
}

int Lane::Build(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const uint8_t* remote) {
    if (params.output_format < FMT_NATIVE || params.output_format > FMT_RGB_PLANAR)
        return Fail(kInvalidParameter, "unknown output format");
    h_images_.assign(size_t(n), ImageDesc{});
    h_outputs_.assign(size_t(n), OutputDesc{});
    h_img_cta0_.assign(size_t(n) + 1, 0);
    h_img_dctile0_.assign(size_t(n) + 1, 0);
    h_k2_tile0_.assign(size_t(n) + 1, 0);
    h_k3_tile0_.assign(size_t(n) + 1, 0);
    for (auto& v : h_k2s_tile0_) v.assign(size_t(n) + 1, 0);
    h_scale_.assign(size_t(n), 1);
    h_fused_.clear();
    h_tile_img_.clear();
    h_tile_img_w_.clear();
    h_gather_.assign(size_t(n), GatherItem{});
    h_lut_ptrs_.clear();
    h_lut_specs_.clear();
    h_lut_hashes_.clear();
    h_qtables_.assign(size_t(n) * 3 * 64, 1);
    stats_ = BatchStats();

    uint64_t total_clean = 0;   // entropy-coded bytes as uploaded (destuffing removes well under 1 % of them)
    for (int i = 0; i < n; i++) {
        if (!streams[i]) return Fail(kInvalidParameter, "null stream handle in batch");
        const ParsedJpeg& p = streams[i]->parsed();
        if (!p.valid) return Fail(kBadJpeg, "stream handle holds no successfully parsed JPEG");
        if (p.support_status != kSuccess) {
            return Fail(p.support_status, "unsupported or inconsistent JPEG");
        }
        if (!streams[i]->raw().host) return Fail(kOutOfMemory, "no staging memory for the scan");
        total_clean += p.raw_bytes;
    }
    // Subsequence size. Long subsequences amortise the speculative re-decodes (with interleaved
    // 4:2:0 data a wrong start state needs about one MCU to re-synchronise); short ones only pay
    // off when the whole batch is too small to occupy the GPU otherwise.
    int S = EnvInt("ROCJPEG_B200_SUBSEQ", 0);
    // (measured: a lone 1920x1080 picture, 0.47 MB of scan, decodes 11 % faster with 64-byte subsequences
    // - every pass of the latency-bound synchronisation is half as long; the 15 MB batch of 256 pictures,
    // one full wave of CTAs at 128 bytes, is 20 % slower in that stage with 64)
    if (S != 32 && S != 64 && S != 128) S = (total_clean >= (2u << 20)) ? 128 : (total_clean >= (48u << 10)) ? 64 : 32;
    stats_.sub_bytes = S;
    // Halo: subsequences before a CTA's own that it re-decodes so that the state entering its first own
    // one is already synchronised. Small pictures (at most a wave of CTAs, the kernel as slow as its slowest
    // CTA): 768 bytes' worth, after which the verifying round has nothing left to repair on the benchmark
    // batches - a repair costs a staging and a chain of decodes, 15-20 us; large ones (many waves,
    // throughput bound): two subsequences, every halo thread is 0.8 % more CTAs.
    int halo = EnvInt("ROCJPEG_B200_HALO", 0);
    if (halo < 1 || halo > 16) halo = (n > 0 && total_clean / uint64_t(n) >= (512u << 10)) ? 2 : std::min(16, 768 / S);
    const uint32_t owned = uint32_t(kK1Threads - halo);

    any_direct_ = false;
    needs_planes_ = false;
    const bool direct_ok = EnvInt("ROCJPEG_B200_NO_DIRECT", 0) == 0;
    const bool fuse_ok = EnvInt("ROCJPEG_B200_NO_FUSE", 0) == 0;
    uint32_t k23tile = 0, k23tile_w = 0;
    const bool warp_ok = EnvInt("ROCJPEG_B200_NO_WARP_FUSE", 0) == 0;
    k2_needed_ = false;
    uint64_t scan_off = 0, raw_off = 0, blk = 0, plane_off = 0, ent = 0, sub = 0;
    uint32_t dctile = 0, k2tile = 0, k3tile = 0, max_pairs = 1, max_sub = 0, k0tile = 0, nseg_total = 0;
    uint32_t k2stile[kScaledKernels] = {};
    all_pinned_ = true;
    // Upload plan. Streams that lie close together in ONE page-locked allocation (the caller's arena of files, or
    // the staging pool's slab) are uploaded by a single copy that takes the few bytes between them along: the copy
    // engine moves such a run at the full PCIe rate (48-50 GB/s measured against 33 GB/s for the gather kernel's
    // reads of mapped memory) and occupies no SM. The device-side layout of a run mirrors the host's.
    h_runs_.clear();
    std::vector<uint64_t> plan_off(size_t(n), 0);
    bool merged = EnvInt("ROCJPEG_B200_NO_MERGE", 0) == 0 && n > 0;
    if (merged) {
        constexpr size_t kMaxGap = 16u << 10;
        uint64_t payload = 0, moved = 0;
        CopyRun run = {};
        uintptr_t run_range = 0, run_range_end = 0;
        auto close_run = [&]() {
            if (!run.src) return;
            run.nbytes = std::min<size_t>(run.nbytes, run_range_end - reinterpret_cast<uintptr_t>(run.src));   // never read past the allocation
            moved += run.nbytes;
            h_runs_.push_back(run);
        };
        for (int i = 0; i < n && merged; i++) {
            const RawScan& rs = streams[i]->raw();
            if (!rs.dev || rs.range_base == 0) { merged = false; break; }
            const uint32_t skip = uint32_t(reinterpret_cast<uintptr_t>(rs.dev) & 15u);
            const uint8_t* start = rs.host - skip;
            const size_t up_bytes = AlignUp(size_t(skip) + rs.nbytes, 16);
            payload += up_bytes;
            if (reinterpret_cast<uintptr_t>(start) < rs.range_base) { merged = false; break; }
            if (run.src && rs.range_base == run_range && start >= run.src + run.nbytes && size_t(start - (run.src + run.nbytes)) <= kMaxGap) {
                plan_off[size_t(i)] = run.dst_off + uint64_t(start - run.src);
                run.nbytes = size_t(start - run.src) + up_bytes;
            } else {
                const uint64_t next = run.src ? AlignUp(size_t(run.dst_off) + run.nbytes + 16, 128) : 0;
                close_run();
                run.src = start;
                run.dst_off = next;
                run.nbytes = up_bytes;
                run_range = rs.range_base;
                run_range_end = rs.range_base + rs.range_size;
                plan_off[size_t(i)] = next;
            }
        }
        close_run();
        // worth it when a handful of copies replace the gather kernel (a copy call costs the host 2-3 us) and the
        // bytes between the streams are a small share of what is moved
        if (merged && (h_runs_.size() > std::max<size_t>(4, size_t(n) / 16) || moved > payload + payload / 4 + (64u << 10))) merged = false;
        if (!merged) h_runs_.clear();
    }
    h_k0_tile0_.assign(size_t(n) + 1, 0);
    h_needed_segments_.assign(size_t(n), 1);
    for (int i = 0; i < n; i++) {
        const ParsedJpeg& p = streams[i]->parsed();
        ImageDesc& im = h_images_[size_t(i)];
        // scale 1/d: the output is ceil(W/d) x ceil(H/d); crop rectangle and destinations are in those units
        const int d = dsts[i].scale_denom;
        if (!ValidScale(d)) return Fail(kInvalidParameter, "scale denominator must be 1, 2, 4 or 8");
        h_scale_[size_t(i)] = d;
        const int out_w = (p.width + d - 1) / d, out_h = (p.height + d - 1) / d;
        im.width = p.width; im.height = p.height; im.ncomp = p.ncomp; im.css = p.css;
        im.mcus_x = p.mcus_x; im.mcus_y = p.mcus_y; im.bpm = p.bpm; im.restart_interval = p.restart_interval;
        im.total_mcus = p.mcus_x * p.mcus_y;
        int k = 0;
        for (int c = 0; c < 3; c++) {
            const bool have = c < p.ncomp;
            const int H = !have ? 0 : (p.ncomp == 1 ? 1 : p.hs[c]), V = !have ? 0 : (p.ncomp == 1 ? 1 : p.vs[c]);
            im.hs[c] = H; im.vs[c] = V;
            im.blocks_w[c] = have ? p.blocks_w[c] : 0;
            im.blocks_h[c] = have ? p.blocks_h[c] : 0;
            im.comp_first_blk[c] = k;
            // (DC table, AC table) pair of the component: K1 keeps each pair's two tables back to back
            int pair = -1;
            if (have) {
                for (int q = 0; q < im.npairs; q++)
                    if (im.pair_dc[q] == p.td[c] && im.pair_ac[q] == kHuffIds + p.ta[c]) pair = q;
                if (pair < 0) {
                    pair = im.npairs++;
                    im.pair_dc[pair] = uint8_t(p.td[c]);
                    im.pair_ac[pair] = uint8_t(kHuffIds + p.ta[c]);
                }
            }
            for (int b = 0; b < H * V && k < kMaxBlocksPerMcu; b++, k++) {
                im.mcu_comp[k] = uint8_t(c);
                im.mcu_dc[k] = uint8_t(p.td[c]);
                im.mcu_ac[k] = uint8_t(kHuffIds + p.ta[c]);
                im.mcu_pair[k] = uint8_t(pair);
            }
            im.qt_index[c] = i * 3 + c;
            im.comp_bits = 0;
            for (int b = 0; b < k; b++) im.comp_bits |= uint32_t(im.mcu_comp[b]) << (2 * b);
            if (have) std::memcpy(&h_qtables_[(size_t(i) * 3 + c) * 64], p.qt_natural[p.tq[c]], 128);
        }
        // Huffman table set, de-duplicated across the batch
        int set = -1;
        for (size_t s = 0; s < h_lut_hashes_.size(); s++)
            // same DHT content -> same decoder-form tables (they are a pure function of the four specs);
            // comparing the 1 KiB of specs instead of the 14 KiB LUTs keeps this loop off the e2e profile
            if (h_lut_hashes_[s] == p.lut_hash && std::memcmp(h_lut_specs_[s]->dc, p.dc, sizeof(p.dc)) == 0 &&
                std::memcmp(h_lut_specs_[s]->ac, p.ac, sizeof(p.ac)) == 0) {
                set = int(s);
                break;
            }
        if (set < 0) {
            set = int(h_lut_ptrs_.size());
            h_lut_ptrs_.push_back(&streams[i]->lut());
            h_lut_specs_.push_back(&p);
            h_lut_hashes_.push_back(p.lut_hash);
        }
        im.lut_set = set;
        max_pairs = std::max(max_pairs, uint32_t(im.npairs));
        max_sub = std::max(max_sub, (streams[i]->lut().sub_used + 3u) & ~3u);
        // entropy-coded data: uploaded raw (whole 16-byte vectors around it), destuffed on the device (k0_destuff.cu)
        const RawScan& rs = streams[i]->raw();
        const uint8_t* src = rs.dev ? rs.dev : rs.host;
        im.raw_skip = uint32_t(reinterpret_cast<uintptr_t>(src) & 15u);
        im.raw_len = rs.nbytes;
        const uint32_t up_bytes = uint32_t(AlignUp(size_t(im.raw_skip) + rs.nbytes, 16));
        if (merged) raw_off = plan_off[size_t(i)];
        im.raw_off = raw_off;
        h_gather_[size_t(i)] = GatherItem{src - im.raw_skip, raw_off, up_bytes, 0u};
        all_pinned_ = all_pinned_ && rs.dev != nullptr;
        raw_off += AlignUp(size_t(up_bytes) + 16, 128);   // (merged: the arena's end is taken from the last run below)
        im.k0_tile0 = k0tile;
        h_k0_tile0_[size_t(i)] = k0tile;
        k0tile += std::max<uint32_t>(1u, uint32_t((size_t(im.raw_skip) + rs.nbytes + kK0TileBytes - 1) / kK0TileBytes));
        im.data_off = scan_off;
        im.seg0 = nseg_total;
        im.nseg = p.nseg;
        {   // restart intervals the frame needs (p.nseg is bounded by what the bytes can hold)
            const uint64_t mcus = uint64_t(im.total_mcus);
            h_needed_segments_[size_t(i)] = p.restart_interval > 0 ? uint32_t((mcus + uint32_t(p.restart_interval) - 1) / uint32_t(p.restart_interval)) : 1u;
        }
        nseg_total += p.nseg;
        const uint64_t clean_cap = CleanCapacity(rs.nbytes, p.nseg, uint32_t(S));
        scan_off += clean_cap;
        im.sub0 = uint32_t(sub);
        im.nsub = uint32_t(clean_cap / uint32_t(S));
        sub = AlignUp(sub + im.nsub, owned);
        if (sub > 0x7FFFFFFFull || nseg_total > 0x7FFFFFFFu) return Fail(kNotSupported, "batch too large for one decode call");
        h_img_cta0_[size_t(i)] = im.sub0 / owned;
        // Region of interest + restart markers: a restart interval is an independent unit (predictors
        // reset), so the intervals whose MCU rows lie wholly outside the crop rectangle are not entropy-
        // decoded at all (same ROI rule as below: src/rocjpeg_decoder.cpp:126-131). The interval in front
        // of the first wanted one is kept: the first block of an interval finds where its coefficient
        // entries begin in the record of the block before it.
        im.seg_keep_lo = 0;
        im.seg_keep_hi = 0xFFFFFFFFu;
        {
            const uint32_t cw = uint32_t(int(params.crop_right) - int(params.crop_left));
            const uint32_t chh = uint32_t(int(params.crop_bottom) - int(params.crop_top));
            if (p.restart_interval > 0 && cw > 0 && chh > 0 && cw <= uint32_t(out_w) && chh <= uint32_t(out_h) &&
                params.crop_top >= 0 && params.crop_bottom <= out_h && im.mcus_y > 0) {
                const int mcu_h = 8 * std::max(1, p.ncomp == 1 ? 1 : p.vmax) / d;   // MCU rows in output rows
                const uint64_t row_lo = uint64_t(params.crop_top / mcu_h), row_hi = uint64_t((params.crop_bottom - 1) / mcu_h);
                const uint64_t ri = uint64_t(p.restart_interval);
                const uint64_t k_lo = row_lo * uint64_t(im.mcus_x) / ri, k_hi = ((row_hi + 1) * uint64_t(im.mcus_x) - 1) / ri;
                im.seg_keep_lo = uint32_t(k_lo > 0 ? k_lo - 1 : 0);
                im.seg_keep_hi = uint32_t(std::min<uint64_t>(k_hi, 0xFFFFFFFFull));
            }
        }
        // coefficients, DC tiles
        im.blk0 = blk;
        im.nblocks = uint32_t(im.total_mcus) * uint32_t(p.bpm);
        blk += im.nblocks;
        // entry arena: every entry consumes at least min_entry_bits of the scan, and a block holds at most 64
        im.ent0 = ent;
        // (+7 padding entries per subsequence: every thread's run is rounded up to whole 32-byte stores)
        const uint64_t ent_cap = uint64_t(rs.nbytes) * 8 / p.min_entry_bits + 7 * (uint64_t(im.nsub) + 1) + 64;
        if (ent_cap > 0xFFFFFF00ull) return Fail(kNotSupported, "scan too large for one picture");
        im.ent_cap = uint32_t(ent_cap);
        ent += (uint64_t(im.ent_cap) + 63) & ~uint64_t(63);
        im.dc_tile0 = dctile;
        h_img_dctile0_[size_t(i)] = dctile;
        dctile += uint32_t((im.total_mcus + kDcTileMcus - 1) / kDcTileMcus);
        // planes + IDCT tiles
        // (a picture at scale 1/d has planes of (blocks_w * 8/d) x (blocks_h * 8/d) samples and its tiles in the kernel of that scale)
        h_k2_tile0_[size_t(i)] = k2tile;
        for (int s = 0; s < kScaledKernels; s++) h_k2s_tile0_[s][size_t(i)] = k2stile[s];
        uint32_t& idct_tiles = d == 1 ? k2tile : k2stile[ScaleIndex(d)];
        const int bs = 8 / d;   // samples per block row and column
        for (int c = 0; c < p.ncomp; c++) {
            im.plane_pitch[c] = uint32_t(AlignUp(size_t(p.blocks_w[c]) * bs, 64));
            im.plane_off[c] = plane_off;
            plane_off += AlignUp(size_t(im.plane_pitch[c]) * size_t(p.blocks_h[c]) * bs, 256);
            idct_tiles += uint32_t((p.blocks_w[c] + 31) / 32) * uint32_t(p.blocks_h[c]);
            stats_.plane_bytes += uint64_t(p.blocks_w[c]) * p.blocks_h[c] * uint64_t(bs * bs);
        }
        // output job. ROI rule: src/rocjpeg_decoder.cpp:126-131 (unsigned widths).
        OutputDesc& od = h_outputs_[size_t(i)];
        const uint32_t rw = uint32_t(int(params.crop_right) - int(params.crop_left));
        const uint32_t rh = uint32_t(int(params.crop_bottom) - int(params.crop_top));
        od.x0 = od.y0 = 0;
        od.w = out_w;
        od.h = out_h;
        if (rw > 0 && rh > 0 && rw <= uint32_t(out_w) && rh <= uint32_t(out_h)) {
            if (params.crop_left < 0 || params.crop_top < 0 || params.crop_right > out_w || params.crop_bottom > out_h)
                return Fail(kInvalidParameter, "crop rectangle lies outside the picture");
            od.x0 = params.crop_left; od.y0 = params.crop_top; od.w = int32_t(rw); od.h = int32_t(rh);
        }
        od.fmt = params.output_format;
        for (int c = 0; c < 4; c++) {
            od.dst[c] = dsts[i].channel[c];
            od.dst_pitch[c] = dsts[i].pitch[c];
        }
        // Planar formats without a crop need no output stage: the IDCT stage stores the planes straight
        // into the caller's channels (4:2:2 / 4:2:0 NATIVE are interleaved surfaces and keep their tiles).
        const bool whole = od.x0 == 0 && od.y0 == 0 && od.w == out_w && od.h == out_h;
        const bool planar = od.fmt == FMT_Y || od.fmt == FMT_YUV_PLANAR ||
                            (od.fmt == FMT_NATIVE && (p.css == CSS_444 || p.css == CSS_440 || p.css == CSS_411 || p.css == CSS_400));
        od.direct = (whole && planar && direct_ok && !(remote && remote[i])) ? 1 : 0;
        // Whole-picture RGB / RGB_PLANAR: IDCT and colour conversion in one kernel, the planes never leave shared memory
        // (full size only: a scaled picture goes reduced-size IDCT -> plane arena -> output stage)
        od.fused = (d == 1 && whole && fuse_ok && (od.fmt == FMT_RGB || od.fmt == FMT_RGB_PLANAR) && h_fused_.size() < 65535) ? 1 : 0;
        const bool tiles = !od.direct && !od.fused;
        od.tiles_x = tiles ? uint32_t((od.w + kK3TileW - 1) / kK3TileW) : 0u;
        od.tiles_y = tiles ? uint32_t((od.h + kK3TileH - 1) / kK3TileH) : 0u;
        any_direct_ = any_direct_ || od.direct || od.fused || !whole;   // the plane arena is then incomplete: the tap re-runs the IDCT
        needs_planes_ = needs_planes_ || tiles;
        k2_needed_ = k2_needed_ || (!od.fused && d == 1);
        if (od.fused) {
            FusedImage fi = {};
            fi.ent0 = im.ent0; fi.blk0 = im.blk0; fi.ent_cap = im.ent_cap;
            for (int c = 0; c < 3; c++) fi.dst[c] = od.dst[c];
            fi.dpitch = od.dst_pitch[0];
            fi.width = p.width; fi.height = p.height; fi.css = p.css; fi.fmt = od.fmt;
            fi.ncomp = p.ncomp; fi.bpm = p.bpm; fi.mcus_x = p.mcus_x;
            int hmax = 1, vmax = 1;
            for (int c = 0; c < p.ncomp; c++) { hmax = std::max(hmax, im.hs[c]); vmax = std::max(vmax, im.vs[c]); }
            fi.vmax = vmax;
            fi.mpt = kK3TileW / (8 * hmax);
            fi.tiles_x = uint32_t((p.width + kK3TileW - 1) / kK3TileW);
            // destination rows all 4-byte aligned (every row takes the register path): the warp-per-column kernel
            bool aligned = (od.dst_pitch[0] & 3u) == 0;
            for (int c = 0; c < (od.fmt == FMT_RGB ? 1 : 3); c++) aligned = aligned && (reinterpret_cast<uintptr_t>(od.dst[c]) & 3u) == 0;
            aligned = aligned && warp_ok && (fi.mpt / 8) * p.bpm <= 16;   // a warp's MCUs hold at most 16 blocks (k23_fused.cu)
            // a destination on another GPU: the strip kernel's rows cross NVLink as 256-pixel segments, the warp kernel's as 32-byte ones
            if (remote && remote[i]) aligned = false;
            fi.tile0 = aligned ? k23tile_w : k23tile;
            fi.sx = p.css == CSS_411 ? 2 : (p.css == CSS_422 || p.css == CSS_420) ? 1 : 0;
            fi.sy = (p.css == CSS_440 || p.css == CSS_420) ? 1 : 0;
            uint32_t off = 0;
            for (int c = 0; c < p.ncomp; c++) {
                fi.H[c] = uint8_t(im.hs[c]); fi.V[c] = uint8_t(im.vs[c]); fi.first_blk[c] = uint8_t(im.comp_first_blk[c]);
                fi.hshift[c] = uint8_t(im.hs[c] == 4 ? 2 : im.hs[c] == 2 ? 1 : 0);
                fi.qidx[c] = uint32_t(im.qt_index[c]);
                fi.pitch[c] = uint32_t(8 * fi.mpt * im.hs[c]);
                fi.base[c] = off;
                fi.comp_info[c] = uint32_t(fi.H[c]) | (uint32_t(fi.V[c]) << 8) | (uint32_t(fi.first_blk[c]) << 16) | (uint32_t(fi.hshift[c]) << 24);
                off += c == 0 ? 16u * kK3TileW : 8u * kK3TileW;   // plane capacities in the kernel's shared memory
            }
            const uint32_t ntiles = fi.tiles_x * uint32_t(p.mcus_y);
            std::vector<uint32_t>& list = aligned ? h_tile_img_w_ : h_tile_img_;
            for (uint32_t r = 0; r < uint32_t(p.mcus_y); r++) list.insert(list.end(), fi.tiles_x, uint32_t(h_fused_.size()) | (r << 16));   // picture | MCU row << 16
            h_fused_.push_back(fi);
            (aligned ? k23tile_w : k23tile) += ntiles;
            stats_.fused_blocks += im.nblocks;
        }
        od.tile0 = k3tile;
        h_k3_tile0_[size_t(i)] = k3tile;
        k3tile += od.tiles_x * od.tiles_y;
        stats_.output_bytes += OutputBytes(p.css, od.fmt, od.w, od.h);
    }
    h_img_cta0_[size_t(n)] = uint32_t(sub / owned);
    h_k0_tile0_[size_t(n)] = k0tile;
    h_img_dctile0_[size_t(n)] = dctile;
    h_k2_tile0_[size_t(n)] = k2tile;
    for (int s = 0; s < kScaledKernels; s++) h_k2s_tile0_[s][size_t(n)] = k2stile[s];
    h_k3_tile0_[size_t(n)] = k3tile;
    scan_bytes_ = scan_off;
    raw_bytes_ = raw_off;
    if (!h_runs_.empty()) raw_bytes_ = AlignUp(size_t(h_runs_.back().dst_off) + h_runs_.back().nbytes + 16, 128);
    nseg_total_ = nseg_total;
    coef_blocks_ = blk;
    entry_count_ = ent;
    plane_bytes_ = plane_off;
    nsub_total_ = sub;
    stats_.scan_bytes = total_clean;
    stats_.blocks = blk;
    stats_.subsequences = sub;

    k1_ = K1Args{};
    k1_.nimages = n;
    k1_.total_ctas = uint32_t(sub / owned);
    k1_.halo = halo;
    k0_ = K0Args{};
    k0_.nimages = n;
    k0_.total_tiles = k0tile;
    k0_.sub_bytes = S;
    {
        uint32_t most_tiles = 0;
        for (int i = 0; i < n; i++) most_tiles = std::max(most_tiles, h_k0_tile0_[size_t(i) + 1] - h_k0_tile0_[size_t(i)]);
        k0_.inline_scan = (most_tiles <= 32u && EnvInt("ROCJPEG_B200_NO_INLINE_SCAN", 0) == 0) ? 1 : 0;
    }
    k1_.rec_fill_vecs = uint32_t((blk * sizeof(BlockRec) + 15) / 16);   // the slab leaves 256 bytes behind every array
    k1_.lut_smem_bytes = max_pairs * 2u * uint32_t(kFastSize) * 4u + max_sub * 4u;
    k1_.total_dc_tiles = dctile;
    k1_.sub_bytes = S;
    {
        uint32_t most = 0;
        for (int i = 0; i < n; i++) most = std::max(most, h_img_cta0_[size_t(i) + 1] - h_img_cta0_[size_t(i)]);
        k1_.inline_scan = (most <= 32u && EnvInt("ROCJPEG_B200_NO_INLINE_SCAN", 0) == 0) ? 1 : 0;
        k1_.fusable = most <= uint32_t(std::max(0, EnvInt("ROCJPEG_B200_K1_FUSE_CTAS", 256))) ? 1 : 0;
        uint32_t most_mcus = 0;
        for (int i = 0; i < n; i++) most_mcus = std::max(most_mcus, uint32_t(h_images_[size_t(i)].total_mcus));
        // one CTA per picture: a lone picture of 8000 MCUs is faster through the tiled kernels (0.013 against 0.06 ms
        // for 1920x1080), a lane full of such pictures keeps every SM busy either way and saves two launches
        const int dc_limit = EnvInt("ROCJPEG_B200_DC_IMAGE_MCUS", n >= 16 ? 2 * kDcImageMaxMcus : kDcImageMaxMcus);
        k1_.dc_image = (most_mcus <= uint32_t(std::max(0, dc_limit)) && EnvInt("ROCJPEG_B200_NO_DC_IMAGE", 0) == 0) ? 1 : 0;
    }
    k2_ = K2Args{};
    k2_.nimages = n;
    k2_.total_tiles = k2tile;
    for (int s = 0; s < kScaledKernels; s++) {
        k2s_[s] = K2Args{};
        k2s_[s].nimages = n;
        k2s_[s].total_tiles = k2stile[s];
    }
    k3_ = K3Args{};
    k3_.nimages = n;
    k3_.total_tiles = k3tile;
    k23_ = K23Args{};
    k23_.nimages = n;
    k23_.total_tiles = k23tile;
    k23_.total_tiles_w = k23tile_w;
    return kSuccess;
}

// Descriptor block: one pinned host buffer mirrored by one device buffer, one copy.
struct Lane::Layout {
    size_t images, outputs, cta0, k0tile0, dctile0, k2tile0, k2stile0[kScaledKernels], k3tile0, fused, tile_img, tile_img_w, gather, luts, qtables, total;
};

int Lane::Upload(cudaStream_t up, UploadTurn turn) {
    TurnGuard guard(turn);
    if (up == nullptr) up = stream_;
    const size_t n = h_images_.size();
    Layout L;
    size_t o = 0;
    auto place = [&](size_t bytes) { size_t at = o; o = AlignUp(o + bytes, 256); return at; };
    L.images = place(n * sizeof(ImageDesc));
    L.outputs = place(n * sizeof(OutputDesc));
    L.cta0 = place((n + 1) * 4);
    L.k0tile0 = place((n + 1) * 4);
    L.dctile0 = place((n + 1) * 4);
    L.k2tile0 = place((n + 1) * 4);
    for (int s = 0; s < kScaledKernels; s++) L.k2stile0[s] = place((n + 1) * 4);
    L.k3tile0 = place((n + 1) * 4);
    L.fused = place(h_fused_.size() * sizeof(FusedImage));
    L.tile_img = place(h_tile_img_.size() * 4);
    L.tile_img_w = place(h_tile_img_w_.size() * 4);
    L.gather = place(n * sizeof(GatherItem));
    L.luts = place(h_lut_ptrs_.size() * sizeof(HuffLutSet));
    L.qtables = place(h_qtables_.size() * 2);
    L.total = o;
    uint8_t* h = h_desc_.Reserve(L.total);
    if (!h) return Fail(kOutOfMemory, "descriptor staging");
    std::memcpy(h + L.images, h_images_.data(), n * sizeof(ImageDesc));
    std::memcpy(h + L.outputs, h_outputs_.data(), n * sizeof(OutputDesc));
    std::memcpy(h + L.cta0, h_img_cta0_.data(), (n + 1) * 4);
    std::memcpy(h + L.k0tile0, h_k0_tile0_.data(), (n + 1) * 4);
    std::memcpy(h + L.dctile0, h_img_dctile0_.data(), (n + 1) * 4);
    std::memcpy(h + L.k2tile0, h_k2_tile0_.data(), (n + 1) * 4);
    for (int s = 0; s < kScaledKernels; s++) std::memcpy(h + L.k2stile0[s], h_k2s_tile0_[s].data(), (n + 1) * 4);
    std::memcpy(h + L.k3tile0, h_k3_tile0_.data(), (n + 1) * 4);
    std::memcpy(h + L.fused, h_fused_.data(), h_fused_.size() * sizeof(FusedImage));
    std::memcpy(h + L.tile_img, h_tile_img_.data(), h_tile_img_.size() * 4);
    std::memcpy(h + L.tile_img_w, h_tile_img_w_.data(), h_tile_img_w_.size() * 4);
    std::memcpy(h + L.gather, h_gather_.data(), n * sizeof(GatherItem));
    for (size_t s = 0; s < h_lut_ptrs_.size(); s++) std::memcpy(h + L.luts + s * sizeof(HuffLutSet), h_lut_ptrs_[s], sizeof(HuffLutSet));
    std::memcpy(h + L.qtables, h_qtables_.data(), h_qtables_.size() * 2);
    desc_bytes_ = L.total;

    // One device allocation per lane (grow-only): the first call of a handle - the only one the
    // reference's perf sample times when it is given a single batch - pays one cudaMalloc, not fifteen.
    // The plane arena is separate and only exists when some image needs the output stage.
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t at = off; off = AlignUp(off + bytes + 256, 256); return at; };
    const size_t o_desc = carve(L.total), o_raw = carve(raw_bytes_ + 512), o_scan = carve(scan_bytes_ + 512),
                 o_segments = carve(size_t(nseg_total_) * sizeof(SegmentDesc)), o_tile_sum = carve(size_t(k0_.total_tiles) * 16),
                 o_tile_carry = carve(size_t(k0_.total_tiles) * 16), o_status = carve(n * sizeof(ScanStatus)), o_entries = carve(entry_count_ * 4),
                 o_blkrec = carve(coef_blocks_ * sizeof(BlockRec)), o_nnz = carve(nsub_total_ * 4), o_state = carve(nsub_total_ * 4),
                 o_used = carve(nsub_total_ * 4), o_subseg = carve(nsub_total_ * 4), o_cta_entries = carve(size_t(k1_.total_ctas) * 4),
                 o_cta_partial = carve(size_t(k1_.total_ctas) * 8), o_cta_carry = carve(size_t(k1_.total_ctas) * 8), o_cta_flag = carve(size_t(k1_.total_ctas) * 8 + 4),
                 o_cta_dc = carve(size_t(k1_.total_ctas) * 32),
                 o_dc_partial = carve(size_t(k1_.total_dc_tiles) * 12), o_dc_carry = carve(size_t(k1_.total_dc_tiles) * 12),
                 o_end = carve(0);
    (void)o_end;
    RJB_CUDA(d_slab_.Reserve(off));
    if (needs_planes_) RJB_CUDA(d_planes_.Reserve(plane_bytes_ + 512));
    if (!h_counters_.Reserve(256 + n * sizeof(ScanStatus))) return Fail(kOutOfMemory, "counter staging");

    uint8_t* base = d_slab_.as<uint8_t>();
    uint8_t* d = base + o_desc;
    k1_.images = reinterpret_cast<const ImageDesc*>(d + L.images);
    k1_.segments = reinterpret_cast<const SegmentDesc*>(base + o_segments);
    k0_.images = k1_.images;
    k0_.segments = reinterpret_cast<SegmentDesc*>(base + o_segments);
    k0_.img_tile0 = reinterpret_cast<const uint32_t*>(d + L.k0tile0);
    k0_.raw = base + o_raw;
    k0_.clean = base + o_scan;
    k0_.tile_sum = reinterpret_cast<uint4*>(base + o_tile_sum);
    k0_.tile_carry = reinterpret_cast<uint4*>(base + o_tile_carry);
    k0_.status = reinterpret_cast<ScanStatus*>(base + o_status);
    k1_.status = k0_.status;
    k1_.img_cta0 = reinterpret_cast<const uint32_t*>(d + L.cta0);
    k1_.img_dctile0 = reinterpret_cast<const uint32_t*>(d + L.dctile0);
    k1_.scan = base + o_scan;
    k1_.luts = reinterpret_cast<const HuffLutSet*>(d + L.luts);
    k1_.state = reinterpret_cast<uint32_t*>(base + o_state);
    k1_.used = reinterpret_cast<uint32_t*>(base + o_used);
    k1_.sub_seg = reinterpret_cast<uint32_t*>(base + o_subseg);
    k1_.cta_partial = reinterpret_cast<uint2*>(base + o_cta_partial);
    k1_.dc_partial = reinterpret_cast<int3*>(base + o_dc_partial);
    k1_.dc_carry = reinterpret_cast<int3*>(base + o_dc_carry);
    k1_.cta_carry = reinterpret_cast<uint2*>(base + o_cta_carry);
    k1_.cta_flag = reinterpret_cast<uint32_t*>(base + o_cta_flag);
    k1_.cta_dc = reinterpret_cast<int4*>(base + o_cta_dc);
    // the batch's counter set is picked at launch time (LaunchAll): the sets alternate
    k1_.entries = reinterpret_cast<uint32_t*>(base + o_entries);
    k1_.blk_rec = reinterpret_cast<BlockRec*>(base + o_blkrec);
    k1_.nnz = reinterpret_cast<uint32_t*>(base + o_nnz);
    k1_.cta_entries = reinterpret_cast<uint32_t*>(base + o_cta_entries);
    k2_.images = k1_.images;
    k2_.outputs = reinterpret_cast<const OutputDesc*>(d + L.outputs);
    k2_.force_planes = 0;
    k2_.img_tile0 = reinterpret_cast<const uint32_t*>(d + L.k2tile0);
    k2_.qtables = reinterpret_cast<const uint16_t*>(d + L.qtables);
    k2_.entries = k1_.entries;
    k2_.blk_rec = k1_.blk_rec;
    k2_.planes = needs_planes_ ? d_planes_.as<uint8_t>() : nullptr;
    for (int s = 0; s < kScaledKernels; s++) {
        const uint32_t tiles = k2s_[s].total_tiles;
        k2s_[s] = k2_;
        k2s_[s].img_tile0 = reinterpret_cast<const uint32_t*>(d + L.k2stile0[s]);
        k2s_[s].total_tiles = tiles;
    }
    k3_.images = k1_.images;
    k3_.outputs = reinterpret_cast<const OutputDesc*>(d + L.outputs);
    k3_.img_tile0 = reinterpret_cast<const uint32_t*>(d + L.k3tile0);
    k3_.planes = k2_.planes;
    k23_.fused = reinterpret_cast<const FusedImage*>(d + L.fused);
    k23_.tile_img = reinterpret_cast<const uint32_t*>(d + L.tile_img);
    k23_.tile_img_w = reinterpret_cast<const uint32_t*>(d + L.tile_img_w);
    k23_.qtables = k2_.qtables;
    k23_.entries = k1_.entries;
    k23_.blk_rec = k1_.blk_rec;

    // Uploads of all lanes go through ONE stream, in lane order: the first chunk gets the whole
    // PCIe link and its kernels start while the next chunks are still in flight.
    guard.Acquire();
    host_ms_[1] = NowMs();
    if (ev_trace_[0]) RJB_CUDA(cudaEventRecord(ev_trace_[0], up));
    RJB_CUDA(cudaMemcpyAsync(d, h, L.total, cudaMemcpyHostToDevice, up));
    stats_.h2d_bytes = L.total;
    for (const GatherItem& g : h_gather_) stats_.h2d_bytes += g.nbytes;
    // Many small pictures: one gather kernel reading the parsers' mapped page-locked buffers (a copy call
    // per picture would cost the host more than the transfer). Few large ones: plain copies, which run on
    // the copy engine at full PCIe rate without occupying SMs.
    const bool use_runs = !h_runs_.empty();
    const bool use_gather = !use_runs && all_pinned_ && h_images_.size() > 4 && raw_bytes_ / h_images_.size() < (256u << 10) &&
                            EnvInt("ROCJPEG_B200_NO_GATHER", 0) == 0;
    tiles_reduced_ = use_gather;
    if (use_gather) {   // ... which also leaves the per-tile prefix elements of the destuffing pass
        RJB_CUDA(LaunchGatherReduce(k0_, reinterpret_cast<const GatherItem*>(d + L.gather), up));
        stats_.kernel_launches++;
    } else if (use_runs) {
        stats_.h2d_bytes = L.total;
        for (const CopyRun& r : h_runs_) {
            RJB_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(k0_.raw) + r.dst_off, r.src, r.nbytes, cudaMemcpyHostToDevice, up));
            stats_.h2d_bytes += r.nbytes;
        }
    } else {
        for (size_t i = 0; i < n; i++)
            RJB_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(k0_.raw) + h_gather_[i].dst_off, h_gather_[i].src, h_gather_[i].nbytes,
                                     cudaMemcpyHostToDevice, up));
    }
    if (ev_trace_[1]) RJB_CUDA(cudaEventRecord(ev_trace_[1], up));
    if (up != stream_) {
        RJB_CUDA(cudaEventRecord(ev_uploaded_, up));
        guard.Release();
        RJB_CUDA(cudaStreamWaitEvent(stream_, ev_uploaded_, 0));
    }
    return kSuccess;
}

int Lane::LaunchAll(bool include_upload, int profiling_, cudaStream_t up, UploadTurn turn) {
    const int rounds = std::min(std::max(EnvInt("ROCJPEG_B200_SYNC_ROUNDS", 2), 1), kMaxSyncRounds);
    // profiling 1: an event after every stage (they sit between the kernels, so neighbouring stages no longer
    // overlap through programmatic dependent launch); 2: only the first and the last event (total time)
    // ROCJPEG_B200_DEBUG_SYNC=1: synchronise after every stage and say which one failed
    static const bool debug_sync = EnvInt("ROCJPEG_B200_DEBUG_SYNC", 0) != 0;
    auto mark = [&](int i) -> cudaError_t {
        if (debug_sync) {
            const cudaError_t e = cudaStreamSynchronize(stream_);
            if (e != cudaSuccess) {
                static const char* const kNames[] = {"(before)", "upload", "destuff", "huffman sync", "huffman write", "dc", "idct", "output"};
                std::cerr << "[rocjpeg_b200] stage '" << kNames[i] << "' failed: " << cudaGetErrorName(e) << std::endl;
                return e;
            }
        }
        const bool want = profiling_ == 1 || (profiling_ == 2 && (i == 0 || i == kStageCount));
        return want ? cudaEventRecord(ev_[i], stream_) : cudaSuccess;
    };
    stats_.kernel_launches = 0;
    // whatever happens below, the lanes queued behind this one on the upload stream get their turn (the guard passes it on
    // when this function leaves before Upload() did), and a failure leaves both counter sets clean for the next call
    struct ExitGuard {
        Lane* lane;
        TurnGuard turn;
        bool ok = false;
        ~ExitGuard() {
            if (!ok && lane->d_counters_.capacity() >= 512) cudaMemsetAsync(lane->d_counters_.as<uint8_t>(), 0, 512, lane->stream_);
        }
    } exit_guard{this, TurnGuard(include_upload ? turn : UploadTurn())};
    RJB_CUDA(mark(0));
    if (include_upload) {
        exit_guard.turn.passed = true;   // Upload() owns the turn from here on (its own guard passes it on)
        int st = Upload(up, turn);
        if (st != kSuccess) return st;
    }
    RJB_CUDA(mark(1));
    // Per-block records start as "never decoded" (8 bytes per block; the entry arena itself is
    // never cleared): blocks a damaged stream does not reach then decode as zero.
    // (round 0 of k1_sync writes the fill, spread over its CTAs - one launch less on the critical path;
    // a batch without any subsequence to decode has no round 0)
    // Counters: two sets; this batch's set was zeroed by the previous batch's write pass (or at creation),
    // its own write pass zeroes the other one - no memset in front of the first kernel.
    k1_.counters = d_counters_.as<uint32_t>() + 64 * counter_set_;
    k1_.counters_next = d_counters_.as<uint32_t>() + 64 * (counter_set_ ^ 1);
    counter_set_ ^= 1;
    if (k1_.total_ctas == 0) {
        RJB_CUDA(cudaMemsetAsync(k1_.blk_rec, 0xFF, coef_blocks_ * sizeof(BlockRec), stream_));
        RJB_CUDA(cudaMemsetAsync(k1_.counters_next, 0, 256, stream_));
    }
    // Counting and write pass of the entropy stage in one kernel when no picture has more than 256 K1 CTAs (k1_huffman.cu:
    // k1_fused); ROCJPEG_B200_NO_K1_FUSE=1 or an explicit ROCJPEG_B200_SYNC_ROUNDS keep the separate kernels.
    const bool k1_fuse_ok = EnvInt("ROCJPEG_B200_NO_K1_FUSE", 0) == 0 && std::getenv("ROCJPEG_B200_SYNC_ROUNDS") == nullptr;
    const bool k1_fused = k1_fuse_ok && k1_.fusable && k1_.total_ctas != 0;
    // ... and, for pictures small enough for dc_image, it integrates the DC differences itself (no DC launch behind it;
    // ROCJPEG_B200_NO_K1_DC=1 keeps it). Not for larger ones: a CTA waits there for the picture's earlier CTAs to finish
    // writing, and with the many CTAs of 4K pictures those waits hold SM slots the next wave needs (c4_dri 3.29 -> 3.65 ms)
    k1_.k1_dc = k1_fused && k1_.dc_image && EnvInt("ROCJPEG_B200_NO_K1_DC", 0) == 0 ? 1 : 0;
    // "published" flags of the CTAs, the ticket counter, the CTAs' DC flags
    if (k1_fused) RJB_CUDA(cudaMemsetAsync(k1_.cta_flag, 0, size_t(k1_.total_ctas) * 8 + 4, stream_));
    // K0: end of slice, destuffing, restart intervals -> clean stream + segment table, all on the device
    if (!(include_upload && tiles_reduced_)) {   // cudaMemcpy upload, or a resident batch run again: the reduction is its own launch
        RJB_CUDA(LaunchK0Reduce(k0_, stream_));
        stats_.kernel_launches++;
    }
    RJB_CUDA(LaunchK0Destuff(k0_, stream_));
    stats_.kernel_launches += k0_.inline_scan ? 1 : 2;
    RJB_CUDA(mark(2));
    if (k1_fused) {
        RJB_CUDA(LaunchK1Fused(k1_, stream_));
        stats_.sync_rounds = 1;   // counters[0] = CTA boundaries that did not hold: Finish() then runs the separate kernels
        RJB_CUDA(mark(3));
    } else {
        for (int r = 0; r < rounds; r++) RJB_CUDA(LaunchK1Sync(k1_, r, stream_));
        stats_.sync_rounds = uint32_t(rounds);
        RJB_CUDA(mark(3));
        RJB_CUDA(LaunchK1Write(k1_, stream_));
    }
    RJB_CUDA(mark(4));
    if (!k1_.k1_dc) RJB_CUDA(LaunchDcScan(k1_, stream_));
    RJB_CUDA(mark(5));
    uint32_t idct_launches = 0;
    {
        const int st = LaunchIdct(false, &idct_launches);
        if (st != kSuccess) return st;
    }
    RJB_CUDA(mark(6));
    RJB_CUDA(LaunchK23Fused(k23_, stream_));
    RJB_CUDA(LaunchK3Output(k3_, stream_));
    RJB_CUDA(mark(7));
    stats_.kernel_launches += (k1_fused ? 1u : uint32_t(rounds) + (k1_.inline_scan ? 1u : 2u)) + (k1_.k1_dc ? 0 : k1_.dc_image ? 1 : 3) + idct_launches +
                              (k23_.total_tiles ? 1 : 0) + (k23_.total_tiles_w ? 1 : 0) +
                              (k3_.total_tiles ? 1 : 0);   // sync rounds, (scan +) write, 0, 1 or 3 DC kernels, IDCT, fused IDCT + output, output
    RJB_CUDA(cudaMemcpyAsync(h_counters_.data(), k1_.counters, 256, cudaMemcpyDeviceToHost, stream_));
    RJB_CUDA(cudaMemcpyAsync(h_counters_.data() + 256, k0_.status, h_images_.size() * sizeof(ScanStatus), cudaMemcpyDeviceToHost, stream_));
    stats_.d2h_bytes = 256 + h_images_.size() * sizeof(ScanStatus);
    if (ev_trace_[2]) RJB_CUDA(cudaEventRecord(ev_trace_[2], stream_));
    host_ms_[2] = NowMs();
    exit_guard.ok = true;
    return kSuccess;
}

int Lane::LaunchIdct(bool force_planes, uint32_t* launches) {
    // (force_planes: the plane tap's re-run, which transforms every picture - fused ones included - into the arena)
    K2Args k2 = k2_;
    k2.force_planes = force_planes ? 1 : 0;
    if (k2_needed_ || force_planes) {
        RJB_CUDA(LaunchK2Idct(k2, stream_));
        if (k2.total_tiles) (*launches)++;
    }
    for (int s = 0; s < kScaledKernels; s++) {
        K2Args ks = k2s_[s];
        ks.force_planes = k2.force_planes;
        RJB_CUDA(LaunchK2Scaled(ks, 2 << s, stream_));
        if (ks.total_tiles) (*launches)++;
    }
    return kSuccess;
}

int Lane::Finish(int profiling_) {
    RJB_CUDA(cudaStreamSynchronize(stream_));
    const uint32_t* cnt = reinterpret_cast<const uint32_t*>(h_counters_.data());
    uint32_t last = stats_.sync_rounds - 1;
    if (cnt[last] != 0) {
        // The stream did not re-synchronise within the rounds launched up front: keep
        // going until a round changes nothing at any CTA boundary, then redo everything
        // downstream of the synchronisation.
        uint32_t guard = 0;
        for (;;) {
            uint32_t slot = std::min<uint32_t>(last + 1, kMaxSyncRounds - 1);
            RJB_CUDA(cudaMemsetAsync(k1_.counters + slot, 0, 4, stream_));
            RJB_CUDA(LaunchK1Sync(k1_, int(slot), stream_));
            RJB_CUDA(cudaMemcpyAsync(h_counters_.data(), k1_.counters, 256, cudaMemcpyDeviceToHost, stream_));
            RJB_CUDA(cudaStreamSynchronize(stream_));
            stats_.sync_rounds++;
            stats_.kernel_launches++;
            last = slot;
            if (cnt[slot] == 0) break;
            if (++guard > k1_.total_ctas + 2) return Fail(kExecutionFailed, "entropy decoder failed to converge");
        }
        RJB_CUDA(cudaMemsetAsync(k1_.blk_rec, 0xFF, coef_blocks_ * sizeof(BlockRec), stream_));
        RJB_CUDA(cudaMemsetAsync(k1_.counters + 2 * kMaxSyncRounds, 0, 4, stream_));   // the first write pass counted its entries already
        RJB_CUDA(LaunchK1ClearShort(k1_, stream_));   // ... and may have reported pictures short that are not
        RJB_CUDA(LaunchK1Write(k1_, stream_));
        RJB_CUDA(LaunchDcScan(k1_, stream_));
        uint32_t idct_launches = 0;
        const int st = LaunchIdct(false, &idct_launches);
        if (st != kSuccess) return st;
        RJB_CUDA(LaunchK23Fused(k23_, stream_));
        RJB_CUDA(LaunchK3Output(k3_, stream_));
        RJB_CUDA(cudaMemcpyAsync(h_counters_.data(), k1_.counters, 256, cudaMemcpyDeviceToHost, stream_));
        RJB_CUDA(cudaMemcpyAsync(h_counters_.data() + 256, k0_.status, h_images_.size() * sizeof(ScanStatus), cudaMemcpyDeviceToHost, stream_));
        RJB_CUDA(cudaStreamSynchronize(stream_));
        stats_.kernel_launches += 8;
    }
    stats_.entries = cnt[2 * kMaxSyncRounds];
    // per-image outcome: what the destuffing pass and the entropy stage found in the bytes
    ScanStatus* st = reinterpret_cast<ScanStatus*>(h_counters_.data() + 256);
    truncated_images_ = 0;
    for (size_t i = 0; i < h_images_.size(); i++) {
        if (st[i].segments_seen < h_needed_segments_[i]) st[i].flags |= kScanMissingIntervals;
        if (st[i].flags & kStatusTruncatedMask) truncated_images_++;
    }
    for (int r = 0; r < kMaxSyncRounds; r++) stats_.decodes_per_round[r] = cnt[kMaxSyncRounds + r];
    if (profiling_) {
        for (int s = 0; s < kStageCount && profiling_ == 1; s++) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev_[s], ev_[s + 1]) == cudaSuccess) stats_.stage_ms[s] = ms;
        }
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ev_[0], ev_[kStageCount]) == cudaSuccess) stats_.total_ms = ms;
        (void)cudaGetLastError();
    }
    return kSuccess;
}

void Lane::PrintTimeline(int index, cudaEvent_t origin, double host_origin_ms) const {
    float t[3] = {-1, -1, -1};
    for (int i = 0; i < 3; i++)
        if (ev_trace_[i] && origin && cudaEventElapsedTime(&t[i], origin, ev_trace_[i]) != cudaSuccess) (void)cudaGetLastError();
    std::fprintf(stderr, "[rocjpeg_b200]   lane %d: %zu images, %zu raw bytes | host: describe %.3f, enqueue %.3f .. %.3f ms | device: upload %.3f .. %.3f, done %.3f ms\n",
                 index, h_images_.size(), raw_bytes_, host_ms_[0] - host_origin_ms, host_ms_[1] - host_origin_ms, host_ms_[2] - host_origin_ms, t[0], t[1], t[2]);
}

// Contiguous split of the batch into chunks of similar entropy-coded size, one per lane.
int Decoder::Split(const StreamParser* const* streams, int n) {
    uint64_t total = 0;
    for (int i = 0; i < n; i++) total += streams[i] ? streams[i]->parsed().raw_bytes : 0;
    int want = EnvInt("ROCJPEG_B200_LANES", 0);
    // about 2 MiB of scan per chunk at least, four chunks at most (every kernel of a chunk is a smaller, less efficient grid:
    // eight chunks cost the 256-picture batch 30 % of its resident throughput) - ROCJPEG_B200_LANES overrides, up to kMaxLanes
    // Large pictures (the call is upload bound, c4: 64 x 2.3 MB): up to eight chunks of 8 MiB or more - the kernels of a
    // chunk of such pictures fill the GPU anyway, and the first chunk's upload, which nothing overlaps, is half as long
    // (c4: 3.80 ms end to end against 4.13 with four chunks).
    if (want <= 0) {
        want = int(std::min<uint64_t>(4, total / (2u << 20)));
        if (n > 0 && total / uint64_t(n) >= (256u << 10)) want = std::max(want, int(std::min<uint64_t>(kMaxLanes, total / (8u << 20))));
    }
    want = std::max(1, std::min(std::min(want, kMaxLanes), n));
    // Chunk sizes as cumulative shares of the scan bytes; ROCJPEG_B200_SPLIT ("30,40,20,10": percentages,
    // one per lane) overrides. Many small pictures: a smaller first and last chunk - the first so that the kernels
    // start early, the last so that the tail behind the final upload is short (c3: 0.82 ms end to end with 20/30/30/20,
    // 0.86 with 30/40/20/10, 0.85 with equal shares; profiles/r03_e2e.md). Few large ones (upload and kernels take
    // about as long): equal shares.
    double cum[kMaxLanes + 1] = {0};
    for (int l = 1; l <= want; l++) cum[l] = double(l) / want;
    if (want == 4 && n > 0 && total / uint64_t(n) < (256u << 10)) {
        cum[1] = 0.20; cum[2] = 0.50; cum[3] = 0.80; cum[4] = 1.0;
    }
    if (const char* sp = std::getenv("ROCJPEG_B200_SPLIT")) {
        double w[kMaxLanes] = {0}, sum = 0;
        int k = 0;
        for (const char* q = sp; *q && k < want;) {
            w[k] = std::max(0.0, std::atof(q));
            sum += w[k++];
            while (*q && *q != ',') q++;
            if (*q == ',') q++;
        }
        if (k == want && sum > 0) {
            double run = 0;
            for (int l = 0; l < want; l++) cum[l + 1] = (run += w[l]) / sum;
        }
    }
    uint64_t acc = 0;
    int lane = 0;
    chunk_first_[0] = 0;
    for (int i = 0; i < n && lane + 1 < want; i++) {
        acc += streams[i] ? streams[i]->parsed().raw_bytes : 0;
        if (double(acc) >= double(total) * cum[lane + 1] && i + 1 < n) chunk_first_[++lane] = i + 1;
    }
    active_lanes_ = lane + 1;
    chunk_first_[active_lanes_] = n;
    return active_lanes_;
}

int Decoder::BuildAll(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, bool launch, const uint8_t* remote) {
    // validate the whole batch before anything is launched: an error leaves every destination untouched
    for (int i = 0; i < n; i++) {
        if (!streams[i]) return Fail(kInvalidParameter, "null stream handle in batch");
        const ParsedJpeg& p = streams[i]->parsed();
        if (!p.valid) return Fail(kBadJpeg, "stream handle holds no successfully parsed JPEG");
        if (p.support_status != kSuccess) {
            if (p.support_status == kNotSupported)
                std::cerr << "[ERR]  {Decode}  The JPEG image (chroma subsampling / layout / size) is not supported!" << std::endl;
            return Fail(p.support_status, "unsupported or inconsistent JPEG");
        }
        const int d = dsts[i].scale_denom;
        if (!ValidScale(d)) return Fail(kInvalidParameter, "scale denominator must be 1, 2, 4 or 8");
        const int out_w = (p.width + d - 1) / d, out_h = (p.height + d - 1) / d;   // the crop rectangle is in output units
        const uint32_t rw = uint32_t(int(params.crop_right) - int(params.crop_left));
        const uint32_t rh = uint32_t(int(params.crop_bottom) - int(params.crop_top));
        if (rw > 0 && rh > 0 && rw <= uint32_t(out_w) && rh <= uint32_t(out_h) &&
            (params.crop_left < 0 || params.crop_top < 0 || params.crop_right > out_w || params.crop_bottom > out_h))
            return Fail(kInvalidParameter, "crop rectangle lies outside the picture");
    }
    if (params.output_format < FMT_NATIVE || params.output_format > FMT_RGB_PLANAR)
        return Fail(kInvalidParameter, "unknown output format");
    Split(streams, n);
    for (int l = 0; l < active_lanes_; l++) {
        const int st = lanes_[l].Create(device_id_, sm_count_, l < 4);
        if (st != kSuccess) return Fail(st, lanes_[l].last_error());
    }
    // Optionally one submitter per lane (ROCJPEG_B200_SUBMIT_THREADS=1): the caller's thread takes lane 0,
    // helper threads the others; uploads are enqueued in lane order, everything else in parallel. Off by
    // default: it cuts the host's submit time from 0.22 to 0.09 ms on the 256-image batch, but the call is
    // bound by the device (upload + pipeline), so the wall time does not move (profiles/r01e_e2e.md).
    const bool threaded = active_lanes_ > 1 && EnvInt("ROCJPEG_B200_SUBMIT_THREADS", 0) != 0;
    std::atomic<int> turn{0};
    int status[kMaxLanes] = {};
    // Pageable input: the parse only reserved page-locked staging; the bytes are copied now, chunk by chunk ahead of each
    // chunk's upload, by a few helper threads (one core copies 16 GB/s, a third of what the upload moves).
    bool any_pending = false;
    for (int i = 0; i < n && !any_pending; i++) any_pending = streams[i]->staging_pending();
    auto stage = [&](int l) {
        const int first = chunk_first_[l], cnt = chunk_first_[l + 1] - first;
        const int threads = std::min(std::max(1, EnvInt("ROCJPEG_B200_COPY_THREADS", 4)), std::min(cnt, kMaxLanes));
        if (threads <= 1) {
            for (int i = first; i < first + cnt; i++) streams[i]->EnsureStaged();
            return;
        }
        if (!pool_) pool_.reset(new SubmitPool(kMaxLanes - 1));
        pool_->Run(threads, [&](int t) {
            for (int i = first + t; i < first + cnt; i += threads) streams[i]->EnsureStaged();
        });
    };
    auto submit = [&](int l) {
        DeviceGuard guard(device_id_);
        Lane& lane = lanes_[l];
        const int first = chunk_first_[l], cnt = chunk_first_[l + 1] - first;
        UploadTurn ut;
        ut.turn = threaded ? &turn : nullptr;
        ut.mine = l;
        lane.set_host_mark(0, NowMs());
        int st = lane.Build(streams + first, cnt, params, dsts + first, remote ? remote + first : nullptr);
        if (st == kSuccess) st = launch ? lane.LaunchAll(true, profiling_, upload_stream_, ut) : lane.Upload(upload_stream_, ut);
        else TurnGuard pass(ut);   // never reached the upload: pass the turn on
        status[l] = st;
    };
    if (threaded) {
        for (int l = 0; l < active_lanes_ && any_pending; l++) stage(l);
        if (!pool_) pool_.reset(new SubmitPool(kMaxLanes - 1));
        pool_->Run(active_lanes_, submit);
    } else {
        for (int l = 0; l < active_lanes_; l++) {
            if (any_pending) stage(l);
            submit(l);
            if (status[l] != kSuccess) break;
        }
    }
    for (int l = 0; l < active_lanes_; l++) {
        if (status[l] != kSuccess) {
            for (int k = 0; k < active_lanes_; k++) lanes_[k].Sync();   // do not leave work in flight behind an error (the failed lane's included)
            return Fail(status[l], lanes_[l].last_error());
        }
    }
    return kSuccess;
}

int Decoder::FinishAll() {
    int status = kSuccess;
    uint32_t truncated = 0;
    for (int l = 0; l < active_lanes_; l++) {
        int st = lanes_[l].Finish(profiling_);
        if (st != kSuccess && status == kSuccess) status = Fail(st, lanes_[l].last_error());
        truncated += lanes_[l].truncated_images();
    }
    Aggregate();
    stats_.truncated_images = truncated;
    // Every picture of the batch has been decoded as far as its bytes go (missing blocks are zero: grey); a scan that
    // ended before its last block makes the call report BAD_JPEG - the VCN path reports a failed surface as an error
    // too (src/rocjpeg_vaapi_decoder.cpp:846-868) - and rocJpegB200GetImageStatus tells which pictures and why.
    if (status == kSuccess && truncated != 0 && strict_status_)
        status = Fail(kBadJpeg, std::to_string(truncated) + " picture(s) of the batch ended before their last block (truncated or damaged scan)");
    return status;
}

void Decoder::Aggregate() {
    stats_ = BatchStats();
    stats_.lanes = active_lanes_;
    for (int l = 0; l < active_lanes_; l++) {
        const BatchStats& s = lanes_[l].stats();
        for (int i = 0; i < kStageCount; i++) stats_.stage_ms[i] += s.stage_ms[i];
        stats_.sync_rounds = std::max(stats_.sync_rounds, s.sync_rounds);
        for (int r = 0; r < kMaxSyncRounds; r++) stats_.decodes_per_round[r] += s.decodes_per_round[r];
        stats_.scan_bytes += s.scan_bytes;
        stats_.blocks += s.blocks;
        stats_.entries += s.entries;
        stats_.subsequences += s.subsequences;
        stats_.plane_bytes += s.plane_bytes;
        stats_.fused_blocks += s.fused_blocks;
        stats_.output_bytes += s.output_bytes;
        stats_.h2d_bytes += s.h2d_bytes;
        stats_.d2h_bytes += s.d2h_bytes;
        stats_.kernel_launches += s.kernel_launches;
        stats_.sub_bytes = std::max(stats_.sub_bytes, s.sub_bytes);
        if (profiling_) {   // wall time on the device: first event of the first lane to the last event of any lane
            float ms = 0;
            if (cudaEventElapsedTime(&ms, lanes_[0].first_event(), lanes_[l].last_event()) == cudaSuccess)
                stats_.total_ms = std::max(stats_.total_ms, ms);
            (void)cudaGetLastError();
        }
    }
}

int Decoder::Decode(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts) {
    std::lock_guard<std::mutex> lock(mutex_);
    if (!initialized_) return Fail(kNotInitialized, "decoder not initialised");
    if (!streams || !dsts || n < 0) return kInvalidParameter;
    if (n == 0) return kSuccess;
    sharded_ = false;
    if (!peers_.empty() && n >= 2) return DecodeSharded(streams, n, params, dsts);
    DeviceGuard guard(device_id_);
    prepared_ = false;
    const auto t0 = std::chrono::steady_clock::now();
    int st = BuildAll(streams, n, params, dsts, true);
    if (st != kSuccess) return st;
    const auto t1 = std::chrono::steady_clock::now();
    st = FinishAll();
    const auto t2 = std::chrono::steady_clock::now();
    stats_.host_submit_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
    stats_.host_wait_ms = std::chrono::duration<float, std::milli>(t2 - t1).count();
    if (TraceLevel()) {
        std::cerr << "[rocjpeg_b200] decode n=" << n << " lanes=" << active_lanes_ << " submit_ms=" << stats_.host_submit_ms
                  << " wait_ms=" << stats_.host_wait_ms << std::endl;
        const double origin = std::chrono::duration<double, std::milli>(t0.time_since_epoch()).count();
        for (int l = 0; l < active_lanes_ && TraceLevel() >= 2; l++) lanes_[l].PrintTimeline(l, lanes_[0].trace_origin(), origin);
    }
    prepared_ = (st == kSuccess) || (st == kBadJpeg && stats_.truncated_images != 0);   // a truncated picture still leaves a decoded batch behind
    return st;
}

int Decoder::Submit(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts, const uint8_t* remote) {
    DeviceGuard guard(device_id_);
    prepared_ = false;
    return BuildAll(streams, n, params, dsts, true, remote);
}

int Decoder::Wait() {
    DeviceGuard guard(device_id_);
    int st = FinishAll();
    prepared_ = (st == kSuccess) || (st == kBadJpeg && stats_.truncated_images != 0);
    return st;
}

int Decoder::DecodeSharded(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts) {
    const auto t0 = std::chrono::steady_clock::now();
    const int ndev = 1 + int(peers_.size());
    // validate first so that an error leaves every destination untouched on every device
    std::vector<uint64_t> cost(static_cast<size_t>(n), 0);
    for (int i = 0; i < n; i++) {
        if (!streams[i]) return Fail(kInvalidParameter, "null stream handle in batch");
        const ParsedJpeg& p = streams[i]->parsed();
        if (!p.valid) return Fail(kBadJpeg, "stream handle holds no successfully parsed JPEG");
        if (p.support_status != kSuccess) return Fail(p.support_status, "unsupported or inconsistent JPEG");
        cost[size_t(i)] = p.raw_bytes;
    }
    // Where does each destination live? An image whose buffer is on one of the peer devices this handle drives is
    // decoded there (its pixels never cross a link); the others - buffers on the handle's own device, the reference
    // samples' case - are dealt by the longest-processing-time rule over all devices, and those that land on a peer
    // are delivered over NVLink.
    std::vector<int> fixed(static_cast<size_t>(n), -1), owner(static_cast<size_t>(n), 0);
    uintptr_t range_base = 0;
    size_t range_size = 0;
    int range_dev = -1;
    for (int i = 0; i < n; i++) {
        const uintptr_t ptr = reinterpret_cast<uintptr_t>(dsts[i].channel[0]);
        if (!(range_size != 0 && ptr >= range_base && ptr - range_base < range_size))   // not in the allocation asked about last
            range_dev = DeviceOfPointer(dsts[i].channel[0], &range_base, &range_size);
        const int dev = range_dev;
        for (int d = 1; d < ndev; d++)
            if (dev == peers_[size_t(d - 1)]->device_id()) fixed[size_t(i)] = d;
        if (dev >= 0 && dev != device_id_ && fixed[size_t(i)] < 0)
            return Fail(kInvalidParameter, "destination buffer on a device this handle does not drive");
        owner[size_t(i)] = fixed[size_t(i)] >= 0 ? fixed[size_t(i)] : 0;
    }
    shard_dev_.assign(size_t(n), 0);
    shard_local_.assign(size_t(n), 0);
    PlanShardsPinned(cost.data(), fixed.data(), n, ndev, shard_dev_.data());
    std::vector<std::vector<const StreamParser*>> sub_streams(static_cast<size_t>(ndev));
    std::vector<std::vector<DestImage>> sub_dsts(static_cast<size_t>(ndev));
    std::vector<std::vector<uint8_t>> sub_remote(static_cast<size_t>(ndev));
    for (int i = 0; i < n; i++) {
        const size_t d = size_t(shard_dev_[size_t(i)]);
        shard_local_[size_t(i)] = int(sub_streams[d].size());
        sub_streams[d].push_back(streams[i]);
        sub_dsts[d].push_back(dsts[i]);
        sub_remote[d].push_back(uint8_t(int(d) != owner[size_t(i)] ? 1 : 0));
    }
    // enqueue everything on every device - one submitter thread per device, the caller's thread taking
    // this handle's device - then join: the devices run concurrently
    int status = kSuccess;
    std::vector<char> submitted(static_cast<size_t>(ndev), 0);
    std::vector<int> sub_status(static_cast<size_t>(ndev), kSuccess);
    auto submit = [&](int d) {
        if (sub_streams[size_t(d)].empty()) return;
        Decoder* dec = d == 0 ? this : peers_[size_t(d - 1)].get();
        sub_status[size_t(d)] = dec->Submit(sub_streams[size_t(d)].data(), int(sub_streams[size_t(d)].size()), params, sub_dsts[size_t(d)].data(),
                                             sub_remote[size_t(d)].data());
        submitted[size_t(d)] = sub_status[size_t(d)] == kSuccess ? 1 : 0;
    };
    if (!shard_pool_) shard_pool_.reset(new SubmitPool(ndev - 1));
    shard_pool_->Run(ndev, submit);
    for (int d = 0; d < ndev; d++)
        if (sub_status[size_t(d)] != kSuccess && status == kSuccess)
            status = Fail(sub_status[size_t(d)], (d == 0 ? this : peers_[size_t(d - 1)].get())->last_error());
    const auto t1 = std::chrono::steady_clock::now();
    BatchStats total;
    total.devices = 0;
    for (int d = 0; d < ndev; d++) {
        if (!submitted[size_t(d)]) continue;
        Decoder* dec = d == 0 ? this : peers_[size_t(d - 1)].get();
        const int st = dec->Wait();
        if (st != kSuccess && status == kSuccess) status = Fail(st, dec->last_error());
        const BatchStats& s = dec->stats_;
        for (int i = 0; i < kStageCount; i++) total.stage_ms[i] += s.stage_ms[i];
        total.total_ms = std::max(total.total_ms, s.total_ms);
        total.sync_rounds = std::max(total.sync_rounds, s.sync_rounds);
        for (int r = 0; r < kMaxSyncRounds; r++) total.decodes_per_round[r] += s.decodes_per_round[r];
        total.scan_bytes += s.scan_bytes;
        total.blocks += s.blocks;
        total.entries += s.entries;
        total.truncated_images += s.truncated_images;
        total.subsequences += s.subsequences;
        total.plane_bytes += s.plane_bytes;
        total.fused_blocks += s.fused_blocks;
        total.output_bytes += s.output_bytes;
        total.h2d_bytes += s.h2d_bytes;
        total.d2h_bytes += s.d2h_bytes;
        total.kernel_launches += s.kernel_launches;
        total.sub_bytes = std::max(total.sub_bytes, s.sub_bytes);
        total.lanes += s.lanes;
        total.devices++;
    }
    const auto t2 = std::chrono::steady_clock::now();
    stats_ = total;
    stats_.host_submit_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
    stats_.host_wait_ms = std::chrono::duration<float, std::milli>(t2 - t1).count();
    sharded_ = (status == kSuccess) || (status == kBadJpeg && total.truncated_images != 0);
    if (status != kSuccess) prepared_ = false;
    return status;
}

int Decoder::Prepare(const StreamParser* const* streams, int n, const DecodeParams& params, const DestImage* dsts) {
    std::lock_guard<std::mutex> lock(mutex_);
    if (!initialized_) return Fail(kNotInitialized, "decoder not initialised");
    if (!streams || !dsts || n <= 0) return kInvalidParameter;
    DeviceGuard guard(device_id_);
    prepared_ = false;
    int st = BuildAll(streams, n, params, dsts, false);
    if (st != kSuccess) return st;
    for (int l = 0; l < active_lanes_; l++) {
        st = lanes_[l].Sync();
        if (st != kSuccess) return Fail(st, lanes_[l].last_error());
    }
    prepared_ = true;
    return kSuccess;
}

int Decoder::Run() {
    std::lock_guard<std::mutex> lock(mutex_);
    if (!initialized_ || !prepared_) return Fail(kNotInitialized, "no prepared batch");
    DeviceGuard guard(device_id_);
    for (int l = 0; l < active_lanes_; l++) {
        int st = lanes_[l].LaunchAll(false, profiling_, nullptr);
        if (st != kSuccess) return Fail(st, lanes_[l].last_error());
    }
    return FinishAll();
}

Lane* Decoder::Locate(int image, int* local) {
    if (sharded_) {
        if (image < 0 || size_t(image) >= shard_dev_.size()) return nullptr;
        const int d = shard_dev_[size_t(image)];
        if (d > 0) return peers_[size_t(d - 1)]->Locate(shard_local_[size_t(image)], local);
        image = shard_local_[size_t(image)];
    }
    if (!prepared_ || image < 0 || image >= chunk_first_[active_lanes_]) return nullptr;
    int l = 0;
    while (image >= chunk_first_[l + 1]) l++;
    *local = image - chunk_first_[l];
    return &lanes_[l];
}

int Decoder::CopyCoefficients(int image, int16_t* host_out, size_t count) {
    std::lock_guard<std::mutex> lock(mutex_);
    int local = 0;
    Lane* lane = host_out ? Locate(image, &local) : nullptr;
    if (!lane) return kInvalidParameter;
    return lane->CopyCoefficients(local, host_out, count);
}

int Decoder::CopyPlanes(int image, uint8_t* host_out, size_t count) {
    std::lock_guard<std::mutex> lock(mutex_);
    int local = 0;
    Lane* lane = host_out ? Locate(image, &local) : nullptr;
    if (!lane) return kInvalidParameter;
    return lane->CopyPlanes(local, host_out, count);
}

int Decoder::CopySegment(int image, uint32_t segment, uint8_t* host_out, size_t capacity, uint32_t* nbytes) {
    std::lock_guard<std::mutex> lock(mutex_);
    int local = 0;
    Lane* lane = nbytes ? Locate(image, &local) : nullptr;
    if (!lane) return kInvalidParameter;
    return lane->CopySegment(local, segment, host_out, capacity, nbytes);
}

int Decoder::GetScanStatus(int image, ScanStatus* out) {
    std::lock_guard<std::mutex> lock(mutex_);
    int local = 0;
    Lane* lane = out ? Locate(image, &local) : nullptr;
    if (!lane) return kInvalidParameter;
    return lane->GetScanStatus(local, out);
}

int Lane::GetScanStatus(int image, ScanStatus* out) const {
    if (image < 0 || size_t(image) >= h_images_.size()) return kInvalidParameter;
    *out = reinterpret_cast<const ScanStatus*>(h_counters_.data() + 256)[image];   // read back with the counters at the end of the call
    return kSuccess;
}

int Lane::CopySegment(int image, uint32_t segment, uint8_t* host_out, size_t capacity, uint32_t* nbytes) {
    if (image < 0 || size_t(image) >= h_images_.size()) return kInvalidParameter;
    const ImageDesc& im = h_images_[size_t(image)];
    if (segment >= im.nseg) return kInvalidParameter;
    SegmentDesc sd;
    RJB_CUDA(cudaStreamSynchronize(stream_));
    RJB_CUDA(cudaMemcpy(&sd, k1_.segments + im.seg0 + segment, sizeof(sd), cudaMemcpyDeviceToHost));
    *nbytes = sd.nbytes;
    if (host_out) {
        if (capacity < sd.nbytes) return kInvalidParameter;
        if (sd.data_off + sd.nbytes > scan_bytes_) return Fail(kExecutionFailed, "segment table entry outside the scan arena");
        if (sd.nbytes) RJB_CUDA(cudaMemcpy(host_out, k1_.scan + sd.data_off, sd.nbytes, cudaMemcpyDeviceToHost));
    }
    return kSuccess;
}

int Lane::CopyCoefficients(int image, int16_t* host_out, size_t count) {
    if (image < 0 || size_t(image) >= h_images_.size() || !host_out) return kInvalidParameter;
    const ImageDesc& im = h_images_[size_t(image)];
    size_t need = 0;
    for (int c = 0; c < im.ncomp; c++) need += size_t(im.blocks_w[c]) * im.blocks_h[c] * 64;
    if (count < need) return kInvalidParameter;
    // densify the sparse stream on the host: decode-order blocks of 64 int16, natural order
    static const uint8_t kZz[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    std::vector<int16_t> tmp(size_t(im.nblocks) * 64, 0);
    std::vector<BlockRec> recs(im.nblocks);
    std::vector<uint32_t> ents(im.ent_cap);
    RJB_CUDA(cudaMemcpy(recs.data(), k1_.blk_rec + im.blk0, recs.size() * sizeof(BlockRec), cudaMemcpyDeviceToHost));
    RJB_CUDA(cudaMemcpy(ents.data(), k1_.entries + im.ent0, ents.size() * 4, cudaMemcpyDeviceToHost));
    for (size_t b = 0; b < recs.size(); b++) {
        uint32_t e0 = b ? recs[b - 1].end : 0u, e1 = recs[b].end;   // a block's entries begin where its predecessor's end
        if (e0 == kNoEntry || e1 == kNoEntry || e1 < e0 || e1 - e0 > 0xFFFFu || e1 > im.ent_cap) e0 = e1 = 0;   // as K2
        for (uint32_t k = e0; k < e1; k++) tmp[b * 64 + kZz[CoefEntryPos(ents[k])]] = int16_t(ents[k] & 0xFFFFu);
        tmp[b * 64] = recs[b].dc;   // integrated DC lives in the block's record
    }
    size_t base = 0;
    for (int c = 0; c < im.ncomp; c++) {
        const int H = im.hs[c], V = im.vs[c];
        for (int by = 0; by < im.blocks_h[c]; by++)
            for (int bx = 0; bx < im.blocks_w[c]; bx++) {
                const size_t mcu = size_t(by / V) * size_t(im.mcus_x) + size_t(bx / H);
                const size_t k = size_t(im.comp_first_blk[c] + (by % V) * H + (bx % H));
                std::memcpy(host_out + base + (size_t(by) * im.blocks_w[c] + bx) * 64, &tmp[(mcu * im.bpm + k) * 64], 128);
            }
        base += size_t(im.blocks_w[c]) * im.blocks_h[c] * 64;
    }
    return kSuccess;
}

int Lane::CopyPlanes(int image, uint8_t* host_out, size_t count) {
    if (image < 0 || size_t(image) >= h_images_.size() || !host_out) return kInvalidParameter;
    const ImageDesc& im = h_images_[size_t(image)];
    const size_t bs = size_t(8 / h_scale_[size_t(image)]);   // samples per block row and column
    size_t need = 0;
    for (int c = 0; c < im.ncomp; c++) need += size_t(im.blocks_w[c]) * im.blocks_h[c] * bs * bs;
    if (count < need) return kInvalidParameter;
    if (any_direct_) {   // the planes of this batch went straight to the caller: produce them in the arena for the tap
        RJB_CUDA(cudaStreamSynchronize(stream_));
        RJB_CUDA(d_planes_.Reserve(plane_bytes_ + 512));
        k2_.planes = d_planes_.as<uint8_t>();
        k3_.planes = k2_.planes;
        for (K2Args& k : k2s_) k.planes = k2_.planes;
        uint32_t launches = 0;
        const int st = LaunchIdct(true, &launches);
        if (st != kSuccess) return st;
        RJB_CUDA(cudaStreamSynchronize(stream_));
    }
    size_t base = 0;
    for (int c = 0; c < im.ncomp; c++) {
        const size_t w = size_t(im.blocks_w[c]) * bs, h = size_t(im.blocks_h[c]) * bs;
        RJB_CUDA(cudaMemcpy2D(host_out + base, w, d_planes_.as<uint8_t>() + im.plane_off[c], im.plane_pitch[c], w, h,
                              cudaMemcpyDeviceToHost));
        base += w * h;
    }
    return kSuccess;
}

}  // namespace rjb
