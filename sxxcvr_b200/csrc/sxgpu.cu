// sxgpu.cu -- implementation of the C ABI in include/sxgpu.h (libsxgpu.so).
//
// Host-side responsibilities: pick the widest access the caller's pointers allow, size the
// persistent grid from the SM count and the kernel's occupancy, and -- for host buffers --
// run the H2D / convert / D2H pipeline over a ring of device chunks on three streams.
// There is no CPU implementation of any conversion in this file or anywhere in the product.
#include "../../include/sxgpu.h"

#include "sx_kernels.cuh"
#include "sx_bank.cuh"
#include "sx_iir.cuh"
#include "sx_fir.cuh"
#include "sx_nco.cuh"
#include "sx_chan.cuh"
#include "sx_resident.cuh"
#include "host/par_copy.hpp"
#include "host/worker_pool.hpp"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include <sched.h>

using namespace sx;

// ---------------------------------------------------------------------------------------
// Context
// ---------------------------------------------------------------------------------------
namespace {

constexpr int kRingSlots = 4;

struct HostRing {
    size_t chunk_frames = 0; // capacity of every slot, in frames of 8 bytes per side
    void *d_in[kRingSlots] = {};
    void *d_out[kRingSlots] = {};
    void *h_in[kRingSlots] = {};  // pinned bounce, only allocated for pageable callers
    void *h_out[kRingSlots] = {};
    cudaEvent_t copied_in[kRingSlots] = {};
    cudaEvent_t converted[kRingSlots] = {};
    cudaEvent_t done[kRingSlots] = {};
    bool events = false;
};

// Completion flag of the small-call kernel (flagged_convert_kernel): pinned, device-mapped.
struct alignas(64) SmallFlag {
    volatile unsigned long long done;
};

// One direction of the host-buffer path.  The reference locks per stream (one mutex in each
// AlsaPcm, SoapySX.cpp:373, taken at :878 and :979) so that an RX thread and a TX thread run
// side by side (example/plot_rxtx_response.py:65-77); so does this: each direction has its own
// lock, streams, device ring, bounce threads and small-call machinery, and shares nothing with
// the other but the GPU.
struct HostLane {
    std::mutex mutex;
    cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
    cudaStream_t s_slot[kRingSlots] = {}; // one stream per ring slot (pipeline_mode 2)
    HostRing ring;
    std::unique_ptr<sxhost::ParallelCopier> copier_in, copier_out; // bounce copies of pageable callers
    sxhost::Sidekick retirer;                                      // runs the outbound half of the pipeline
    sxhost::Progress issued, retired;
    std::atomic<int> pipeline_error{0};

    // small synchronous calls
    SmallFlag *flag = nullptr;       // pinned
    unsigned int *d_arrivals = nullptr;
    unsigned long long flag_seq = 0;

    // resident converter (sx_resident.cuh)
    Mailbox *mailbox = nullptr;
    cudaStream_t s_resident = nullptr;
    unsigned long long resident_seq = 0;
};

} // namespace

struct sxgpu_ctx {
    int device = 0;
    cudaDeviceProp prop;
    cudaStream_t stream = nullptr;

    // options
    int64_t rx_variant = 0, tx_variant = 0; // 0 auto (= 4), 1 vec128, 2 vec256, 3 bulk (persistent grids), 4 one tile per CTA
    int64_t unroll = 0;                     // 0 auto (4), else 2/4/8
    int64_t block = 0;                      // 0 auto, threads per CTA
    int64_t ctas_per_sm = 0;                // 0 auto
    int64_t bulk_tile = 0, bulk_stages = 0; // 0 auto
    int64_t bulk_load_policy = 0, bulk_store_policy = 0; // L2 eviction: 0 first, 1 normal, 2 last, 3 unchanged
    int64_t bulk_contiguous = 0;            // 0 round-robin tiles, 1 one contiguous range per CTA
    int64_t host_chunk_frames = 0;          // 0 auto (see pick_chunk_frames)
    int64_t host_chunk_min_frames = 0;      // > 0: chunk sizes ramp up from here and mirror at the end (measured: no gain, r02)
    int64_t host_mode = 0;                  // 0 auto, 1 copy engines, 2 zero-copy
    int64_t small_mode = 0;                 // completion of small calls: 0 auto (= 1), 1 stream sync, 2 host flag
    int64_t host_in_mode = 0;               // pipeline input side: 0 auto (= 1), 1 copy engine, 2 read by the kernel across PCIe
    int64_t host_out_mode = 0;              // pipeline output side: 0 auto (= 1), 1 copy engine, 2 written by the kernel across PCIe
    int64_t bounce_nt = 1;                  // bounce copies use cache-bypassing stores
    int64_t pipeline_mode = 0;              // 0 auto (= 1); 1 = copy-in / compute / copy-out streams chained by events;
                                            // 2 = one stream per ring slot, each chunk's three operations in order on it
    int64_t zero_copy_max_frames = 1 << 18; // measured crossover, profiles/r01_sweep_host_path.json
    int64_t resident_max_frames = 0;        // > 0: blocks up to this size go to the resident converter
    int64_t zero_copy_variant = 1;          // schedule of the zero-copy kernel (1 vec128, 2 vec256, 3 bulk)
    int64_t batch_variant = 0;              // blocks above 4096 frames: 0 auto, 1 = slices of CTAs on vector accesses, 2 = one chunk per CTA, 3 = bulk-async tiles
    int64_t loopback_variant = 0;           // 0 auto (= 2), 1 = vector accesses on a persistent grid, 2 = one tile per CTA, 3 = bulk-async
    int64_t warp_ctas_per_sm = 0;           // grid cap of the warp-per-block / warp-per-stream kernels: N CTAs per SM (persistent), 0 = one CTA per eight blocks
    int64_t bank_split_variant = 0;         // sxgpu_bank_read / _write on large banks: 0 auto (plan + data kernels), 1 = warp-per-stream kernels
    int64_t bank_repeat_variant = 0;        // 0 auto; 1, 2, 4 = K streams per warp round; 100 = 32 per CTA round;
                                            // 201, 202, 204 = K per warp round in registers; 600, 604 = plan + data kernels
    int64_t bounce_threads = 0;             // threads copying a pageable caller's buffer: 0 auto, 1 = the caller alone
    int64_t numa_local_alloc = 1;           // place pinned host memory on the GPU's NUMA node
    int64_t numa_node = -1;                 // read-only: the GPU's NUMA node, -1 unknown / no NUMA

    // CPUs local to the GPU (sysfs local_cpulist of its PCI function); empty set = unknown
    cpu_set_t local_cpus;
    bool have_local_cpus = false;

    std::atomic<uint64_t> resident_launches{0}, resident_calls{0}, flagged_calls{0};
    std::atomic<int> live_banks{0}; // banks keep a pointer to their context
    std::atomic<int> live_dsp{0};   // so do filters, oscillators and channelizers
    bool l2_carveout_set = false;   // sxgpu_bank_repeat_begin sets the persisting-L2 limit once

    // host pipeline: lane 0 serves the RX conversions, lane 1 the TX conversions
    HostLane lanes[2];

    cudaMemPool_t scratch_pool = nullptr; // stream-ordered scratch of the batch entry points

    // statistics scratch
    StatsAcc *d_stats = nullptr;
    StatsAcc *h_stats = nullptr;
    std::mutex stats_mutex;

    // counters
    std::atomic<uint64_t> launches{0}, frames_rx{0}, frames_tx{0}, h2d_bytes{0}, d2h_bytes{0};

    std::mutex err_mutex;
    std::string last_error;
    uint64_t error_serial = 0; // bumped with every new message, see sxgpu_last_error

    // occupancy of each (kernel, block, smem) seen so far: the query costs about a microsecond,
    // which matters when the whole call is a 2 KiB block
    std::mutex occupancy_mutex;
    std::map<std::tuple<const void *, int, size_t>, int> occupancy;

    int fail(cudaError_t e, const char *what)
    {
        std::lock_guard<std::mutex> lock(err_mutex);
        last_error = std::string(what) + ": " + cudaGetErrorString(e);
        error_serial++;
        cudaGetLastError(); // clear the sticky-free error state
        return (e == cudaErrorMemoryAllocation) ? SXGPU_ERR_NOMEM : SXGPU_ERR_CUDA;
    }
    int invalid(const char *what)
    {
        std::lock_guard<std::mutex> lock(err_mutex);
        last_error = what;
        error_serial++;
        return SXGPU_ERR_INVALID;
    }
};

namespace {

// The CUDA stream of a call on ctx or on one of its objects: the caller's, or the context's.
cudaStream_t call_stream(const sxgpu_ctx *ctx, sxgpu_stream stream)
{
    return stream ? static_cast<cudaStream_t>(stream) : ctx->stream;
}

// Which CPUs sit next to this GPU?  Linux publishes it per PCI function; a VM without NUMA
// topology lists every CPU and node -1, and then there is nothing to choose.
void read_gpu_locality(sxgpu_ctx *ctx)
{
    CPU_ZERO(&ctx->local_cpus);
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, ctx->device) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    for (char *c = bdf; *c; c++)
        if (*c >= 'A' && *c <= 'F')
            *c = char(*c - 'A' + 'a'); // sysfs spells the address in lower case
    const std::string base = std::string("/sys/bus/pci/devices/") + bdf + "/";
    if (FILE *f = std::fopen((base + "numa_node").c_str(), "r")) {
        long node = -1;
        if (std::fscanf(f, "%ld", &node) == 1)
            ctx->numa_node = node;
        std::fclose(f);
    }
    if (FILE *f = std::fopen((base + "local_cpulist").c_str(), "r")) {
        // "0-15,64-79": comma-separated CPU numbers and inclusive ranges
        int lo = 0, hi = 0, count = 0;
        for (;;) {
            if (std::fscanf(f, "%d", &lo) != 1)
                break;
            hi = lo;
            int c = std::fgetc(f);
            if (c == '-') {
                if (std::fscanf(f, "%d", &hi) != 1)
                    break;
                c = std::fgetc(f);
            }
            for (int cpu = lo; cpu <= hi && cpu < CPU_SETSIZE; cpu++, count++)
                CPU_SET(cpu, &ctx->local_cpus);
            if (c != ',')
                break;
        }
        std::fclose(f);
        ctx->have_local_cpus = count > 0;
    }
}

// While one of these lives, the calling thread runs only on CPUs next to the GPU, so that
// pages the thread faults in (cudaHostAlloc pins fresh pages in the caller's context) come
// from the GPU's NUMA node and its DMA does not cross the socket interconnect.  The previous
// affinity comes back on destruction; the memory stays where it was placed.
class NearGpu {
public:
    explicit NearGpu(sxgpu_ctx *ctx)
    {
        if (!ctx->numa_local_alloc || !ctx->have_local_cpus)
            return;
        if (sched_getaffinity(0, sizeof saved_, &saved_) != 0)
            return;
        cpu_set_t want;
        CPU_AND(&want, &saved_, &ctx->local_cpus); // never widen what the caller was given
        if (CPU_COUNT(&want) == 0 || CPU_EQUAL(&want, &saved_))
            return;
        bound_ = sched_setaffinity(0, sizeof want, &want) == 0;
    }
    ~NearGpu()
    {
        if (bound_)
            sched_setaffinity(0, sizeof saved_, &saved_);
    }
    NearGpu(const NearGpu &) = delete;
    NearGpu &operator=(const NearGpu &) = delete;

private:
    cpu_set_t saved_;
    bool bound_ = false;
};

} // namespace

#define SX_CUDA(ctx, call)                                                                     \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return (ctx)->fail(e_, #call);                                                     \
    } while (0)

#define SX_TRY(expr)                                                                           \
    do {                                                                                       \
        int r_ = (expr);                                                                       \
        if (r_ != SXGPU_OK)                                                                    \
            return r_;                                                                         \
    } while (0)

namespace {

// ---------------------------------------------------------------------------------------
// Kernel tables
// ---------------------------------------------------------------------------------------
typedef void (*StreamKernel)(const StreamArgs);
typedef void (*BulkKernel)(const BulkArgs);

template <class Op, int FR, int BLOCK> StreamKernel stream_kernel_for_unroll(int unroll)
{
    switch (unroll) {
    case 2: return stream_convert_kernel<Op, FR, 2, BLOCK>;
    case 8: return stream_convert_kernel<Op, FR, 8, BLOCK>;
    default: return stream_convert_kernel<Op, FR, 4, BLOCK>;
    }
}

// Instantiated shapes: FR in {2, 4} x UNROLL in {2, 4, 8} x BLOCK in {256, 512}; the
// frame-at-a-time shape (FR = 1, for pointers whose two sides can never be vector-aligned
// together) exists once.
template <class Op> StreamKernel stream_kernel(int fr, int unroll, int block)
{
    if (fr == 4)
        return block == 512 ? stream_kernel_for_unroll<Op, 4, 512>(unroll)
                            : stream_kernel_for_unroll<Op, 4, 256>(unroll);
    if (fr == 2)
        return block == 512 ? stream_kernel_for_unroll<Op, 2, 512>(unroll)
                            : stream_kernel_for_unroll<Op, 2, 256>(unroll);
    return stream_convert_kernel<Op, 1, 4, 256>;
}

struct BulkShape {
    int tile, stages;
};

template <class Op> BulkKernel bulk_kernel(BulkShape s)
{
    if (s.tile == 4096 && s.stages == 3) return bulk_convert_kernel<Op, 4096, 3>;
    if (s.tile == 3072 && s.stages == 4) return bulk_convert_kernel<Op, 3072, 4>;
    if (s.tile == 2048 && s.stages == 6) return bulk_convert_kernel<Op, 2048, 6>;
    if (s.tile == 2048 && s.stages == 5) return bulk_convert_kernel<Op, 2048, 5>;
    if (s.tile == 2048 && s.stages == 4) return bulk_convert_kernel<Op, 2048, 4>;
    if (s.tile == 2048 && s.stages == 3) return bulk_convert_kernel<Op, 2048, 3>;
    if (s.tile == 1024 && s.stages == 6) return bulk_convert_kernel<Op, 1024, 6>;
    if (s.tile == 1024 && s.stages == 4) return bulk_convert_kernel<Op, 1024, 4>;
    if (s.tile == 512 && s.stages == 4) return bulk_convert_kernel<Op, 512, 4>;
    return nullptr;
}

template <class Op> size_t bulk_smem_bytes(BulkShape s, bool skew = false)
{
    return size_t(s.stages) * (size_t(s.tile) * (Op::kSrcWords + Op::kDstWords) * 4 + (skew ? 16 : 0)) +
           size_t(s.stages) * 8;
}

// The one-frame-out-of-step variant exists for the two default shapes of the CF32 conversions.
template <class Op> BulkKernel bulk_skew_kernel(BulkShape s)
{
    if constexpr (Op::kSrcWords == 2 && Op::kDstWords == 2) {
        if (s.tile == 2048 && s.stages == 4) return bulk_convert_kernel<Op, 2048, 4, true>;
        if (s.tile == 1024 && s.stages == 4) return bulk_convert_kernel<Op, 1024, 4, true>;
    }
    return nullptr;
}

int normalise_unroll(int64_t u)
{
    return (u == 2 || u == 4 || u == 8) ? int(u) : 4;
}

// Persistent grid: enough CTAs to fill every SM at the kernel's occupancy, never more than
// there are tiles of work.
template <class K>
int persistent_grid(sxgpu_ctx *ctx, K kernel, int block, size_t smem, uint64_t work_items)
{
    int per_sm = int(ctx->ctas_per_sm);
    if (per_sm <= 0) {
        std::lock_guard<std::mutex> lock(ctx->occupancy_mutex);
        auto key = std::make_tuple(reinterpret_cast<const void *>(kernel), block, smem);
        auto it = ctx->occupancy.find(key);
        if (it == ctx->occupancy.end()) {
            int occ = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, smem) != cudaSuccess ||
                occ <= 0) {
                cudaGetLastError();
                occ = 1;
            }
            it = ctx->occupancy.emplace(key, occ).first;
        }
        per_sm = it->second;
    }
    uint64_t grid = uint64_t(ctx->prop.multiProcessorCount) * uint64_t(per_sm);
    grid = std::min<uint64_t>(grid, std::max<uint64_t>(work_items, 1));
    return int(grid);
}

// ---------------------------------------------------------------------------------------
// Alignment analysis: the widest access both sides allow, and the head that reaches it
// ---------------------------------------------------------------------------------------
struct Plan {
    int fr = 0;        // frames per access; 0 = word kernel
    uint64_t head = 0; // frames before the aligned middle
};

template <class Op> Plan plan_access(const char *src, const char *dst, uint64_t total, int want_fr)
{
    constexpr uintptr_t SFB = Op::kSrcWords * 4, DFB = Op::kDstWords * 4;
    uintptr_t s = reinterpret_cast<uintptr_t>(src), d = reinterpret_cast<uintptr_t>(dst);
    Plan p;
    if (s % SFB != 0 || d % DFB != 0)
        return p; // frames themselves are misaligned: word accesses
    for (int fr = want_fr; fr >= 1; fr >>= 1) {
        uintptr_t a = (s / SFB) % fr, b = (d / DFB) % fr;
        if (a != b)
            continue; // the two sides can never be vector-aligned at the same frame
        p.fr = fr;
        p.head = std::min<uint64_t>((fr - a) % fr, total);
        return p;
    }
    p.fr = 1;
    return p;
}

// ---------------------------------------------------------------------------------------
// One conversion call on device pointers
// ---------------------------------------------------------------------------------------
template <class Op>
int launch_bulk(sxgpu_ctx *ctx, const char *src, const char *dst_c, uint64_t total, float thr2,
                cudaStream_t st, bool *handled)
{
    char *dst = const_cast<char *>(dst_c);
    constexpr uintptr_t SFB = Op::kSrcWords * 4, DFB = Op::kDstWords * 4;
    constexpr uint64_t G = 16 / (SFB < DFB ? SFB : DFB); // frames per 16 bytes on the narrow side
    *handled = false;

    uint64_t head = 0;
    bool found = false;
    for (; head < G; head++) {
        if ((reinterpret_cast<uintptr_t>(src) + head * SFB) % 16 == 0 &&
            (reinterpret_cast<uintptr_t>(dst) + head * DFB) % 16 == 0) {
            found = true;
            break;
        }
    }

    // Measured (profiles/r01_summary.md): 2048-frame tiles x 4 stages for large blocks; below
    // 2^24 frames the 1024-frame tile spreads the fewer tiles over more SMs.
    // Unequal frame widths (the CS16 / S16 extensions, 12 B/frame): 3072 x 4, measured 0.98-1.04 of
    // the copy peak for all four conversions against 0.78-0.93 on the equal-width default (r02).
    const int big_tile = (SFB == DFB) ? 2048 : 3072;
    BulkShape shape = {int(ctx->bulk_tile ? ctx->bulk_tile : (total >= (uint64_t(1) << 24) ? big_tile : 1024)),
                       int(ctx->bulk_stages ? ctx->bulk_stages : 4)};
    BulkKernel k = nullptr;
    bool skew = false;
    uint64_t mid = 0;
    if (found) {
        if (total < head + G)
            return SXGPU_OK; // too short: the caller falls back to the vector kernel
        mid = (total - head) / G * G;
        k = bulk_kernel<Op>(shape);
        if (!k)
            return ctx->invalid("unsupported bulk_tile/bulk_stages combination");
    } else {
        // No head aligns both sides.  With 8-byte frames on both sides that means they are one
        // frame out of step.  Pick the head (1 or 2 frames) that aligns the DESTINATION and is
        // at least one frame, so that the 8 bytes the skewed loads take in front of the middle
        // are the caller's own frame head-1; and keep at least one frame behind the middle, so
        // that the 8 bytes taken after it are the caller's own too.
        k = bulk_skew_kernel<Op>(shape);
        if (!k || reinterpret_cast<uintptr_t>(src) % 8 || reinterpret_cast<uintptr_t>(dst) % 8)
            return SXGPU_OK;
        head = (reinterpret_cast<uintptr_t>(dst) % 16) ? 1 : 2;
        if (total < head + 3)
            return SXGPU_OK;
        mid = (total - head - 1) / 2 * 2;
        skew = true;
    }
    size_t smem = bulk_smem_bytes<Op>(shape, skew);
    int block = int(ctx->block ? ctx->block : 256);

    BulkArgs a = {src + head * SFB - (skew ? 8 : 0), dst + head * DFB, mid, thr2, int(ctx->bulk_load_policy),
                  int(ctx->bulk_store_policy), int(ctx->bulk_contiguous)};
    uint64_t ntiles = (mid + shape.tile - 1) / shape.tile;
    int grid = persistent_grid(ctx, k, block, smem, ntiles);
    k<<<grid, block, smem, st>>>(a);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;

    // Up to G-1 frames on either side of the 16-byte-aligned middle.
    // (Skewed: 1-2 frames in front and 1-2 behind.)
    uint64_t tail = total - head - mid;
    if (head) {
        StreamArgs e = {src, dst, head, head, 0, thr2};
        stream_convert_kernel<Op, 1, 4, 256><<<1, 256, 0, st>>>(e);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    if (tail) {
        StreamArgs e = {src + (head + mid) * SFB, dst + (head + mid) * DFB, tail, tail, 0, thr2};
        stream_convert_kernel<Op, 1, 4, 256><<<1, 256, 0, st>>>(e);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    *handled = true;
    return SXGPU_OK;
}

template <class Op>
int launch_convert(sxgpu_ctx *ctx, const void *src_v, void *dst_v, uint64_t total, float thr2,
                   int64_t variant, cudaStream_t st)
{
    if (total == 0)
        return SXGPU_OK; // reference: convert_tx_buffer is called with length 0 (:1090)
    const char *src = static_cast<const char *>(src_v);
    char *dst = static_cast<char *>(dst_v);
    if (reinterpret_cast<uintptr_t>(src) % 4 || reinterpret_cast<uintptr_t>(dst) % 4)
        return ctx->invalid("sample buffers must be at least 4-byte aligned");

    // Default (measured, profiles/r02_summary.md section 2): one tile per CTA, CTAs handed out in
    // index order by the hardware.  The addresses in flight then form one compact window that
    // moves through the block, which is what HBM wants to see: 6.9 TB/s against 6.5-6.6 for every
    // persistent schedule (grid-stride vector kernels and the bulk-async ring alike), whose CTAs
    // drift apart as they go.
    if (variant == 0)
        variant = 4;
    if (variant == 4) {
        constexpr bool narrow = Op::kSrcWords != Op::kDstWords; // 12 B/frame: 256 bits on the wide side
        Plan p = plan_access<Op>(src, dst, total, narrow ? 4 : 2);
        if (p.fr >= 2 && total >= p.head + uint64_t(p.fr)) {
            // two accesses per thread in flight; four below 2^21 frames, where fewer, fatter CTAs
            // ramp up faster than more, thinner ones (r02 sweep: 2.0 against 1.4 TB/s at 2^19 frames)
            constexpr int block = 256;
            const int unroll = total < (uint64_t(1) << 21) ? 4 : 2;
            StreamArgs a = {src, dst, total, p.head, (total - p.head) / uint64_t(p.fr), thr2};
            StreamKernel k = stream_kernel<Op>(p.fr, unroll, block);
            uint64_t tiles = (a.nvec + uint64_t(block) * unroll - 1) / (uint64_t(block) * unroll);
            k<<<unsigned(std::min<uint64_t>(tiles, 0x7fffffffu)), block, 0, st>>>(a);
            SX_CUDA(ctx, cudaGetLastError());
            ctx->launches++;
            return SXGPU_OK;
        }
        variant = 3; // the two sides are out of step (or too short): the skewed bulk kernel, then the word kernel
    }
    if (variant == 3) {
        bool handled = false;
        SX_TRY(launch_bulk<Op>(ctx, src, dst, total, thr2, st, &handled));
        if (handled)
            return SXGPU_OK;
        variant = 1;
    }

    Plan p = plan_access<Op>(src, dst, total, variant == 2 ? 4 : 2);
    if (p.fr == 0) {
        const int block = 256;
        uint64_t ctas = (total + block - 1) / block;
        int grid = persistent_grid(ctx, word_convert_kernel<Op>, block, 0, ctas);
        word_convert_kernel<Op><<<grid, block, 0, st>>>(src, dst, total, thr2);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
        return SXGPU_OK;
    }

    int unroll = p.fr == 1 ? 4 : normalise_unroll(ctx->unroll);
    int block = (p.fr != 1 && ctx->block == 512) ? 512 : 256;
    StreamArgs a = {src, dst, total, p.head, (total - p.head) / uint64_t(p.fr), thr2};
    StreamKernel k = stream_kernel<Op>(p.fr, unroll, block);
    uint64_t tiles = (a.nvec + uint64_t(block) * unroll - 1) / (uint64_t(block) * unroll);
    int grid = persistent_grid(ctx, k, block, 0, tiles);
    k<<<grid, block, 0, st>>>(a);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

bool frames_overflow(size_t offset, size_t length)
{
    // 2^60 frames of 8 bytes already overflow a 64-bit byte count.
    const size_t cap = size_t(1) << 60;
    return offset > cap || length > cap || offset + length > cap;
}

template <class Op>
int convert_entry(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                  size_t dest_offset, size_t length, float thr2, int64_t variant,
                  sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (length == 0)
        return SXGPU_OK;
    if (!d_src || !d_dest)
        return ctx->invalid("null sample buffer");
    if (frames_overflow(src_offset, length) || frames_overflow(dest_offset, length))
        return ctx->invalid("offset + length overflows");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const char *src = static_cast<const char *>(d_src) + src_offset * (Op::kSrcWords * 4);
    char *dst = static_cast<char *>(d_dest) + dest_offset * (Op::kDstWords * 4);
    cudaStream_t st = call_stream(ctx, stream);
    return launch_convert<Op>(ctx, src, dst, length, thr2, variant, st);
}

// ---------------------------------------------------------------------------------------
// Host-buffer pipeline
// ---------------------------------------------------------------------------------------
struct HostPtrInfo {
    bool pinned = false;          // page-locked host memory: copy engines can use it in place
    bool on_device = false;       // device (or managed) memory: no PCIe copy needed on this side
    bool foreign_device = false;  // device memory of another GPU
    void *device_alias = nullptr; // address a kernel on this GPU can use for the same memory
};

HostPtrInfo classify_pointer(const sxgpu_ctx *ctx, const void *p)
{
    HostPtrInfo info;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return info; // unknown to CUDA: pageable host memory
    }
    if (attr.type == cudaMemoryTypeHost) {
        info.pinned = true;
        info.device_alias = attr.devicePointer;
    } else if (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) {
        info.on_device = true;
        info.foreign_device = attr.type == cudaMemoryTypeDevice && attr.device != ctx->device;
        info.device_alias = attr.devicePointer;
    }
    return info;
}

// Largest chunk of the copy-engine pipeline.  Measured on B200 / PCIe Gen5 (profiles/
// r01_sweep_host_path.json): about an eighth of the block, between 2 MiB and 32 MiB per
// side, keeps both copy engines busy; the first and last chunks are smaller (plan_chunks).
size_t pick_chunk_frames(const sxgpu_ctx *ctx, size_t length)
{
    if (ctx->host_chunk_frames > 0)
        return size_t(std::max<int64_t>(ctx->host_chunk_frames, 1024));
    // Measured (profiles/r02_summary.md, host path): a quarter of the block, between 1 MiB and
    // 32 MiB per side.  Every queued copy costs ~5 us on the copy engine whatever its size, so
    // chunks below 1 MiB lose more to that than they save in pipeline fill and drain.
    size_t chunk = size_t(1) << 17;
    while (chunk < (size_t(1) << 22) && chunk * 4 < length)
        chunk <<= 1;
    return chunk;
}

int ensure_lane(sxgpu_ctx *ctx, HostLane &lane)
{
    if (!lane.s_h2d) {
        // Ordinary streams (they still run concurrently with each other): a device buffer the
        // caller produced on the default stream is safe to hand to the synchronous calls.
        SX_CUDA(ctx, cudaStreamCreateWithFlags(&lane.s_h2d, cudaStreamDefault));
        SX_CUDA(ctx, cudaStreamCreateWithFlags(&lane.s_comp, cudaStreamDefault));
        SX_CUDA(ctx, cudaStreamCreateWithFlags(&lane.s_d2h, cudaStreamDefault));
        for (int i = 0; i < kRingSlots; i++)
            SX_CUDA(ctx, cudaStreamCreateWithFlags(&lane.s_slot[i], cudaStreamDefault));
    }
    HostRing &r = lane.ring;
    if (!r.events) {
        for (int i = 0; i < kRingSlots; i++) {
            SX_CUDA(ctx, cudaEventCreateWithFlags(&r.copied_in[i], cudaEventDisableTiming));
            SX_CUDA(ctx, cudaEventCreateWithFlags(&r.converted[i], cudaEventDisableTiming));
            SX_CUDA(ctx, cudaEventCreateWithFlags(&r.done[i], cudaEventDisableTiming));
        }
        r.events = true;
    }
    if (!lane.flag) {
        SX_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&lane.flag), sizeof(SmallFlag),
                                   cudaHostAllocMapped | cudaHostAllocPortable));
        lane.flag->done = 0;
        SX_CUDA(ctx, cudaMalloc(reinterpret_cast<void **>(&lane.d_arrivals), sizeof(unsigned int)));
        SX_CUDA(ctx, cudaMemset(lane.d_arrivals, 0, sizeof(unsigned int)));
    }
    return SXGPU_OK;
}

// Ask the lane's resident converter, if one is listening, to leave, and wait until it has.
// Called (lane lock held) before anything that synchronises the whole device.
void resident_stop(sxgpu_ctx *, HostLane &lane)
{
    if (!lane.mailbox || !lane.s_resident)
        return;
    volatile Mailbox *box = lane.mailbox;
    box->quit = 1;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    cudaStreamSynchronize(lane.s_resident);
    box->quit = 0;
}

// Before device memory that kernels may still use is freed: stop the resident converters (each
// would hold the device-wide synchronisation up), then wait for the device.
void quiesce(sxgpu_ctx *ctx)
{
    cudaSetDevice(ctx->device);
    for (HostLane &lane : ctx->lanes) {
        std::lock_guard<std::mutex> lock(lane.mutex);
        resident_stop(ctx, lane);
    }
    cudaDeviceSynchronize();
}

// ---- the lifetime of the DSP objects (filters, oscillators, channelizers) ----------------------
// Their device memory frees itself, so that a create that fails half-way leaves nothing behind and
// a destroy is the object's destructor.
struct CudaFree {
    void operator()(void *p) const { cudaFree(p); }
};
template <class T> using DevPtr = std::unique_ptr<T, CudaFree>;

// `bytes` of device memory holding a copy of the host's src, or zeros when src is NULL, enqueued on
// the context's stream; the create waits for it in dsp_created.
template <class T> cudaError_t dev_upload(sxgpu_ctx *ctx, DevPtr<T> &d, const void *src, size_t bytes)
{
    void *p = nullptr;
    const cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess)
        return e;
    d.reset(static_cast<T *>(p));
    return src ? cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, ctx->stream) : cudaMemsetAsync(p, 0, bytes, ctx->stream);
}

// The end of every DSP object's create: e is the first error of its uploads.  Waits for them, then
// hands the object out and counts it; on an error the object and its memory go.
template <class T> int dsp_created(sxgpu_ctx *ctx, std::unique_ptr<T> &obj, cudaError_t e, const char *what, T **out)
{
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess)
        return ctx->fail(e, what);
    ctx->live_dsp++;
    *out = obj.release();
    return SXGPU_OK;
}

template <class T> int dsp_destroy(T *obj)
{
    if (!obj)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = obj->ctx;
    quiesce(ctx);
    delete obj;
    ctx->live_dsp--;
    return SXGPU_OK;
}

// What get_state / set_state do with a DSP object's device state: `bytes` from src to dst in the
// direction `kind` (dst zeroed when src is NULL) on the call's stream, waited for.
int state_copy(sxgpu_ctx *ctx, void *dst, const void *src, size_t bytes, cudaMemcpyKind kind, sxgpu_stream stream)
{
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const cudaStream_t st = call_stream(ctx, stream);
    if (src)
        SX_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, kind, st));
    else
        SX_CUDA(ctx, cudaMemsetAsync(dst, 0, bytes, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int ensure_ring(sxgpu_ctx *ctx, HostLane &lane, size_t frames, bool bounce_in, bool bounce_out)
{
    SX_TRY(ensure_lane(ctx, lane));
    HostRing &r = lane.ring;
    if (frames > r.chunk_frames) { // grow-only, like the reference's staging vectors (:944, :1087)
        resident_stop(ctx, lane); // cudaFree synchronises the device
        for (int i = 0; i < kRingSlots; i++) {
            if (r.d_in[i]) cudaFree(r.d_in[i]);
            if (r.d_out[i]) cudaFree(r.d_out[i]);
            if (r.h_in[i]) cudaFreeHost(r.h_in[i]);
            if (r.h_out[i]) cudaFreeHost(r.h_out[i]);
            r.d_in[i] = r.d_out[i] = r.h_in[i] = r.h_out[i] = nullptr;
        }
        r.chunk_frames = 0;
        for (int i = 0; i < kRingSlots; i++) {
            SX_CUDA(ctx, cudaMalloc(&r.d_in[i], frames * 8));
            SX_CUDA(ctx, cudaMalloc(&r.d_out[i], frames * 8));
        }
        r.chunk_frames = frames;
    }
    bool missing = false;
    for (int i = 0; i < kRingSlots; i++)
        missing = missing || (bounce_in && !r.h_in[i]) || (bounce_out && !r.h_out[i]);
    if (!missing)
        return SXGPU_OK; // the usual case; nothing below runs per call (NearGpu is two system calls)
    NearGpu near(ctx);
    for (int i = 0; i < kRingSlots; i++) {
        if (bounce_in && !r.h_in[i])
            SX_CUDA(ctx, cudaHostAlloc(&r.h_in[i], r.chunk_frames * 8, cudaHostAllocDefault));
        if (bounce_out && !r.h_out[i])
            SX_CUDA(ctx, cudaHostAlloc(&r.h_out[i], r.chunk_frames * 8, cudaHostAllocDefault));
    }
    return SXGPU_OK;
}

// Hand one small block to the lane's resident converter and wait for it.  `src` and `dst` are
// device-visible addresses of distinct buffers.  Every wait is bounded.
int resident_convert_call(sxgpu_ctx *ctx, HostLane &lane, int op, const void *src, void *dst, size_t length,
                          float thr2)
{
    using clock = std::chrono::steady_clock;
    if (!lane.mailbox) {
        SX_CUDA(ctx, cudaHostAlloc(reinterpret_cast<void **>(&lane.mailbox), sizeof(Mailbox),
                                   cudaHostAllocMapped | cudaHostAllocPortable));
        std::memset(lane.mailbox, 0, sizeof(Mailbox));
        SX_CUDA(ctx, cudaStreamCreateWithFlags(&lane.s_resident, cudaStreamNonBlocking));
    }
    volatile Mailbox *box = lane.mailbox;

    auto ensure_listening = [&]() -> int {
        if (box->alive)
            return SXGPU_OK;
        // No kernel is listening (never started, or it left: idle, lifetime, or asked to).  Wait
        // for the old one to be completely gone, then start a new one and wait until it says so.
        SX_CUDA(ctx, cudaStreamSynchronize(lane.s_resident));
        resident_kernel<<<1, 256, 0, lane.s_resident>>>(lane.mailbox, lane.resident_seq);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
        ctx->resident_launches++;
        auto t0 = clock::now();
        while (!box->alive) {
            if (clock::now() - t0 > std::chrono::seconds(2))
                return ctx->invalid("resident converter did not start");
        }
        return SXGPU_OK;
    };
    SX_TRY(ensure_listening());

    const unsigned long long seq = ++lane.resident_seq;
    unsigned thr2_bits;
    std::memcpy(&thr2_bits, &thr2, sizeof thr2_bits);
    // Fields first, each piece's tag after its fields, `request` last (see Mailbox).
    box->src = static_cast<const char *>(src);
    box->dst = static_cast<char *>(dst);
    std::atomic_thread_fence(std::memory_order_release);
    box->packed = (unsigned long long)(unsigned(length) | (unsigned(op) << 16) | (unsigned(seq & 0x7FFFu) << 17)) |
                  ((unsigned long long)thr2_bits << 32);
    box->request2 = seq;
    std::atomic_thread_fence(std::memory_order_release);
    box->request = seq;

    auto t0 = clock::now();
    unsigned spins = 0;
    while (box->done != seq) {
        if ((++spins & 0xFF) != 0)
            continue;
        if (!box->alive) {
            // The kernel left.  Once it is really gone either it served this request in its last
            // look (done == seq) or it never saw it: then a fresh kernel, started with
            // last_seen = seq - 1, picks it up from the mailbox.
            SX_CUDA(ctx, cudaStreamSynchronize(lane.s_resident));
            if (box->done == seq)
                break;
            lane.resident_seq = seq - 1;
            SX_TRY(ensure_listening());
            lane.resident_seq = seq;
            t0 = clock::now();
        }
        if (clock::now() - t0 > std::chrono::seconds(2))
            return ctx->invalid("resident converter did not answer");
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    ctx->resident_calls++;
    return SXGPU_OK;
}

template <class Op> constexpr int resident_op()
{
    return -1;
}
template <> constexpr int resident_op<RxCf32>()
{
    return 0;
}
template <> constexpr int resident_op<TxCf32>()
{
    return 1;
}

// One small block, one launch, completion through a flag in pinned memory (sx_kernels.cuh,
// flagged_convert_kernel).  `src` and `dst` are device-visible and frame-aligned.
template <class Op>
int flagged_convert_call(sxgpu_ctx *ctx, HostLane &lane, const void *src, void *dst, size_t length, float thr2)
{
    using clock = std::chrono::steady_clock;
    FlaggedArgs a;
    a.block.src = static_cast<const char *>(src);
    a.block.dst = static_cast<char *>(dst);
    a.block.length = length;
    a.block.thr2 = thr2;
    a.block.reserved = 0;
    a.arrivals = lane.d_arrivals;
    a.h_flag = const_cast<unsigned long long *>(&lane.flag->done);
    a.seq = ++lane.flag_seq;
    // 1024 frames per CTA: a period is one CTA, the largest small call one CTA per SM.
    const int grid = int(std::min<uint64_t>((length + 1023) / 1024, uint64_t(ctx->prop.multiProcessorCount)));
    flagged_convert_kernel<Op><<<grid, 256, 0, lane.s_comp>>>(a);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    unsigned spins = 0;
    auto t0 = clock::now();
    while (lane.flag->done != a.seq) {
        if ((++spins & 0xFFF) != 0)
            continue;
        // Every few thousand looks make sure the kernel has not died under us.
        cudaError_t q = cudaStreamQuery(lane.s_comp);
        if (q != cudaSuccess && q != cudaErrorNotReady)
            return ctx->fail(q, "small-call kernel");
        if (q == cudaSuccess && lane.flag->done != a.seq && clock::now() - t0 > std::chrono::milliseconds(100))
            return ctx->invalid("small-call kernel finished without raising its flag");
        if (clock::now() - t0 > std::chrono::seconds(5))
            return ctx->invalid("small-call kernel did not finish");
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    ctx->flagged_calls++;
    return SXGPU_OK;
}

// Threads that share one bounce copy between a pageable caller buffer and pinned staging: half
// of this process's share of the hardware threads, at most eight.  One thread moves 5-7 GB/s
// through the pipeline, eight 32-46, the link behind the staging buffer 46
// (profiles/r01_bench_pageable.json).  Under torchrun the share is 1 / LOCAL_WORLD_SIZE.
unsigned bounce_thread_count(const sxgpu_ctx *ctx)
{
    unsigned threads = unsigned(std::min<int64_t>(ctx->bounce_threads, 64));
    if (threads == 0) {
        // Asked once per process: hardware_concurrency() reads /sys on every call, which a
        // period-sized block (a 2 KiB copy) would pay twice per read+write pair.
        static const unsigned automatic = [] {
            unsigned ranks = 1;
            if (const char *env = std::getenv("LOCAL_WORLD_SIZE"))
                ranks = unsigned(std::max(1, std::atoi(env)));
            return std::max(1u, std::min(8u, std::thread::hardware_concurrency() / (2 * ranks)));
        }();
        threads = automatic;
    }
    return threads;
}

void bounce_copy(sxgpu_ctx *ctx, std::unique_ptr<sxhost::ParallelCopier> &copier, void *dst, const void *src,
                 size_t bytes)
{
    if (bytes < sxhost::ParallelCopier::kMinParallelBytes) { // small: this thread alone, no pool to consult
        if (ctx->bounce_nt)
            sxhost::stream_copy(dst, src, bytes);
        else
            std::memcpy(dst, src, bytes);
        return;
    }
    const unsigned threads = bounce_thread_count(ctx);
    const bool streaming = ctx->bounce_nt != 0;
    if (!copier || copier->helpers() != threads - 1 || copier->streaming() != streaming)
        copier.reset(new sxhost::ParallelCopier(threads - 1, streaming));
    copier->copy(dst, src, bytes);
}

template <class Op> constexpr int lane_of()
{
    return (std::is_same<Op, TxCf32>::value || std::is_same<Op, TxCs16>::value ||
            std::is_same<Op, TxCf32S16>::value)
               ? 1
               : 0;
}

// A gated call (sxgpu_convert_rx_buffer_host_gated): the source buffer is still being filled while
// the conversion runs.  *gate = frames of the block that are in place so far; bit 63 set = that
// count is final (no more will come: the block ends there, possibly short of `length`).
constexpr uint64_t kGateFinal = uint64_t(1) << 63;
// Waits until `need` frames are in place or the count is final; returns the frames that may be
// touched, at most `need`.
inline uint64_t gate_wait(const volatile uint64_t *gate, uint64_t need)
{
    if (!gate)
        return need;
    unsigned spins = 0;
    for (;;) {
        const uint64_t v = __atomic_load_n(const_cast<const uint64_t *>(gate), __ATOMIC_ACQUIRE);
        const uint64_t have = v & ~kGateFinal;
        if (have >= need)
            return need;
        if (v & kGateFinal)
            return have;
        if (++spins > 4000)
            std::this_thread::yield();
    }
}

template <class Op>
int convert_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                 size_t dest_offset, size_t length, float thr2, int64_t variant,
                 const volatile uint64_t *gate = nullptr, size_t *converted = nullptr)
{
    constexpr size_t SFB = Op::kSrcWords * 4, DFB = Op::kDstWords * 4; // frame bytes on each side
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (length == 0)
        return SXGPU_OK;
    if (!h_src || !h_dest)
        return ctx->invalid("null sample buffer");
    if (frames_overflow(src_offset, length) || frames_overflow(dest_offset, length))
        return ctx->invalid("offset + length overflows");
    const char *src = static_cast<const char *>(h_src) + src_offset * SFB;
    char *dst = static_cast<char *>(h_dest) + dest_offset * DFB;

    HostLane &lane = ctx->lanes[lane_of<Op>()];
    std::lock_guard<std::mutex> lock(lane.mutex);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));

    HostPtrInfo si = classify_pointer(ctx, src), di = classify_pointer(ctx, dst);
    if (si.foreign_device || di.foreign_device)
        return ctx->invalid("sample buffer lives on another GPU than the context");
    const uint64_t in_bytes = si.on_device ? 0 : length * SFB, out_bytes = di.on_device ? 0 : length * DFB;

    // One kernel, no queued copies, when the block is already on the device or is small: a
    // period-sized block (256 frames) in pinned host memory is read and written across PCIe by
    // the kernel itself.  Small pageable buffers take the same route through a pinned bounce
    // slot (one memcpy each), which is cheaper than three queued operations.
    const bool both_on_device = si.on_device && di.on_device;
    const bool small = ctx->host_mode == 2 ||
                       (ctx->host_mode == 0 && length <= size_t(ctx->zero_copy_max_frames));
    if (converted)
        *converted = length;
    if (both_on_device || small) {
        if (gate) { // one kernel over the whole block: it has to be there
            length = size_t(gate_wait(gate, length));
            if (converted)
                *converted = length;
            if (length == 0)
                return SXGPU_OK;
        }
        const bool bounce_in = !si.device_alias, bounce_out = !di.device_alias;
        SX_TRY(ensure_ring(ctx, lane, (bounce_in || bounce_out) ? length : 0, bounce_in, bounce_out));
        const void *kernel_in = si.device_alias;
        void *kernel_out = di.device_alias;
        if (bounce_in) {
            bounce_copy(ctx, lane.copier_in, lane.ring.h_in[0], src, length * SFB);
            kernel_in = lane.ring.h_in[0]; // pinned memory is device-addressable at the same address (UVA)
        }
        if (bounce_out)
            kernel_out = lane.ring.h_out[0];
        const bool frame_aligned = reinterpret_cast<uintptr_t>(kernel_in) % SFB == 0 &&
                                   reinterpret_cast<uintptr_t>(kernel_out) % DFB == 0;
        if (resident_op<Op>() >= 0 && !both_on_device && length <= size_t(ctx->resident_max_frames) &&
            length < (size_t(1) << 16) && frame_aligned && kernel_in != kernel_out) {
            SX_TRY(resident_convert_call(ctx, lane, resident_op<Op>(), kernel_in, kernel_out, length, thr2));
        } else if (!both_on_device && ctx->small_mode == 2 && frame_aligned && ctx->host_mode != 2) {
            SX_TRY(flagged_convert_call<Op>(ctx, lane, kernel_in, kernel_out, length, thr2));
        } else {
            SX_TRY(launch_convert<Op>(ctx, kernel_in, kernel_out, length, thr2,
                                      both_on_device ? variant : ctx->zero_copy_variant, lane.s_comp));
            SX_CUDA(ctx, cudaStreamSynchronize(lane.s_comp));
        }
        if (bounce_out)
            bounce_copy(ctx, lane.copier_out, dst, lane.ring.h_out[0], length * DFB);
        ctx->h2d_bytes += in_bytes;
        ctx->d2h_bytes += out_bytes;
        return SXGPU_OK;
    }

    // Copy-engine pipeline over the lane's ring.  A side that is device memory skips its copy:
    // the kernel reads the caller's device buffer, or writes into it, directly.  A side that is
    // pageable host memory is bounced through pinned staging: the inbound copies by this thread
    // (and its helpers) just before each chunk is queued, the outbound copies by the lane's
    // sidekick thread (and its helpers) as each chunk's device-to-host copy completes -- so the
    // two directions' CPU copies, the DMA and the kernels of different chunks all overlap.
    const bool bounce_in = !si.pinned && !si.on_device, bounce_out = !di.pinned && !di.on_device;
    // Up to 2^23 frames the kernel writes its output straight into pinned host memory (posted
    // writes across PCIe run at copy-engine speed) instead of leaving it to a third pipeline stage:
    // one stage less to fill and drain, +5-10 % at 2^19-2^22 frames; beyond that the copy engine is
    // ahead by 2-5 %.  The input side always goes through the copy engine (SM reads of host memory
    // reach 60-70 % of it).
    const bool in_zero_copy = ctx->host_in_mode == 2;
    const bool out_zero_copy = ctx->host_out_mode == 2 || (ctx->host_out_mode == 0 && length <= (size_t(1) << 23));
    const size_t c_max = std::min<size_t>(length, pick_chunk_frames(ctx, length));
    // + 128: the cap is rounded up to 64 frames and the last chunk carries the ragged end (< 64)
    SX_TRY(ensure_ring(ctx, lane, c_max + 128, bounce_in, bounce_out));
    HostRing &r = lane.ring;
    std::vector<sxhost::ChunkSpan> chunks = // (a gated call that ends short trims them as it goes)
        sxhost::plan_chunks(length, size_t(ctx->host_chunk_min_frames), std::min(c_max, r.chunk_frames - 128));
    const size_t nchunks = chunks.size();

    lane.issued.reset();
    lane.retired.reset();
    lane.pipeline_error.store(0);
    const bool use_sidekick = bounce_out;
    if (use_sidekick) {
        lane.retirer.start([ctx, &lane, &r, &chunks, nchunks, dst] {
            if (cudaSetDevice(ctx->device) != cudaSuccess) {
                lane.pipeline_error.store(int(cudaGetLastError()) | 0x10000);
                return;
            }
            for (size_t i = 0; i < nchunks; i++) {
                if (!lane.issued.wait_for(i + 1, lane.pipeline_error))
                    return;
                const int slot = int(i % kRingSlots);
                cudaError_t e = cudaEventSynchronize(r.done[slot]);
                if (e != cudaSuccess) {
                    lane.pipeline_error.store(int(e) | 0x10000);
                    return;
                }
                bounce_copy(ctx, lane.copier_out, dst + chunks[i].first * DFB, r.h_out[slot], chunks[i].frames * DFB);
                lane.retired.publish(i + 1);
            }
        });
    }
    // Whatever happens below, the sidekick is told (pipeline_error) and waited for before return.
    auto finish = [&](int rc) -> int {
        if (use_sidekick) {
            if (rc != SXGPU_OK)
                lane.pipeline_error.store(1);
            lane.retirer.finish();
            const int pe = lane.pipeline_error.load();
            if (rc == SXGPU_OK && (pe & 0x10000))
                rc = ctx->fail(cudaError_t(pe & 0xFFFF), "host pipeline (outbound side)");
        }
        return rc;
    };
    // Two ways to order a chunk's three operations (copy in, convert, copy out).  Chained
    // (default): one stream per kind of operation, events between them.  Per slot: one stream per
    // ring slot, the chunk's operations in order on it and chunk i + K behind chunk i on the same
    // stream, so that the device buffers of a slot need no event at all -- three or four runtime
    // calls per chunk instead of eight.  Measured equal within noise (r02): the pipeline is bound
    // by the copy engines' per-copy cost, not by the calling thread.
    const bool per_slot = ctx->pipeline_mode == 2;
    // Slot i % K is free again once chunk i - K has left it: its device-to-host copy is complete
    // (and, for a pageable destination, bounced out).  With one stream per slot the device side
    // orders itself; only a pinned bounce buffer about to be refilled by the CPU needs the wait.
    auto wait_slot_free = [&](size_t i) -> int {
        if (i < size_t(kRingSlots))
            return SXGPU_OK;
        if (per_slot && !bounce_in && !use_sidekick)
            return SXGPU_OK;
        if (use_sidekick) {
            if (!lane.retired.wait_for(i - kRingSlots + 1, lane.pipeline_error))
                return SXGPU_ERR_CUDA;
            return SXGPU_OK;
        }
        SX_CUDA(ctx, cudaEventSynchronize(r.done[int(i % kRingSlots)]));
        return SXGPU_OK;
    };

    auto issue_all = [&]() -> int {
        for (size_t i = 0; i < nchunks; i++) {
            const int slot = int(i % kRingSlots);
            SX_TRY(wait_slot_free(i));
            const size_t first = chunks[i].first;
            size_t n = chunks[i].frames;
            if (gate) { // the source is still being filled: this chunk's frames, or what the block ends with
                const uint64_t have = gate_wait(gate, first + n);
                if (have < first + n) { // final and short: the block ends inside (or before) this chunk
                    n = have > first ? size_t(have - first) : 0;
                    chunks[i].frames = n;
                    for (size_t j = i + 1; j < nchunks; j++)
                        chunks[j].frames = 0;
                    if (converted)
                        *converted = std::min<size_t>(*converted, first + n);
                }
                if (n == 0) { // nothing of this chunk exists: no work, the slot's events keep their last (completed) state
                    lane.issued.publish(i + 1);
                    continue;
                }
            }

            // Input side: the caller's device buffer as it is; or pinned host memory (the caller's,
            // or the bounce slot) either copied in by the copy engine or read by the kernel itself.
            const void *kernel_in = r.d_in[slot];
            if (si.on_device) {
                kernel_in = static_cast<const char *>(si.device_alias) + first * SFB;
            } else {
                const void *from = src + first * SFB; // host address, for the copy engine
                const void *from_gpu = si.device_alias ? static_cast<const char *>(si.device_alias) + first * SFB : nullptr;
                if (bounce_in) {
                    bounce_copy(ctx, lane.copier_in, r.h_in[slot], src + first * SFB, n * SFB);
                    from = from_gpu = r.h_in[slot]; // cudaHostAlloc memory: one address for both
                }
                if (in_zero_copy && from_gpu) {
                    kernel_in = from_gpu;
                } else if (per_slot) {
                    SX_CUDA(ctx, cudaMemcpyAsync(r.d_in[slot], from, n * SFB, cudaMemcpyHostToDevice, lane.s_slot[slot]));
                } else {
                    SX_CUDA(ctx, cudaMemcpyAsync(r.d_in[slot], from, n * SFB, cudaMemcpyHostToDevice, lane.s_h2d));
                    SX_CUDA(ctx, cudaEventRecord(r.copied_in[slot], lane.s_h2d));
                    SX_CUDA(ctx, cudaStreamWaitEvent(lane.s_comp, r.copied_in[slot], 0));
                }
            }

            // Output side, likewise.
            void *host_to = bounce_out ? r.h_out[slot] : static_cast<void *>(dst + first * DFB);
            void *host_to_gpu = bounce_out          ? r.h_out[slot]
                                : di.device_alias ? static_cast<void *>(static_cast<char *>(di.device_alias) + first * DFB)
                                                  : nullptr;
            const bool kernel_writes_host = !di.on_device && out_zero_copy && host_to_gpu;
            void *kernel_out = di.on_device ? static_cast<void *>(static_cast<char *>(di.device_alias) + first * DFB)
                               : kernel_writes_host ? host_to_gpu
                                                    : r.d_out[slot];
            cudaStream_t s_kernel = per_slot ? lane.s_slot[slot] : lane.s_comp;
            SX_TRY(launch_convert<Op>(ctx, kernel_in, kernel_out, n, thr2, variant, s_kernel));

            if (per_slot) {
                if (!di.on_device && !kernel_writes_host)
                    SX_CUDA(ctx, cudaMemcpyAsync(host_to, r.d_out[slot], n * DFB, cudaMemcpyDeviceToHost, s_kernel));
                // the event is only looked at by the CPU: before a bounce buffer is reused or
                // bounced out, and for the last K chunks at the end of the call
                if (bounce_in || use_sidekick || i + size_t(kRingSlots) >= nchunks)
                    SX_CUDA(ctx, cudaEventRecord(r.done[slot], s_kernel));
            } else if (di.on_device || kernel_writes_host) {
                SX_CUDA(ctx, cudaEventRecord(r.done[slot], lane.s_comp));
            } else {
                SX_CUDA(ctx, cudaEventRecord(r.converted[slot], lane.s_comp));
                SX_CUDA(ctx, cudaStreamWaitEvent(lane.s_d2h, r.converted[slot], 0));
                SX_CUDA(ctx, cudaMemcpyAsync(host_to, r.d_out[slot], n * DFB, cudaMemcpyDeviceToHost, lane.s_d2h));
                SX_CUDA(ctx, cudaEventRecord(r.done[slot], lane.s_d2h));
            }
            lane.issued.publish(i + 1);
        }
        if (!use_sidekick) {
            // The last K chunks are still in flight; events complete in stream order.
            for (size_t i = (nchunks > size_t(kRingSlots) ? nchunks - kRingSlots : 0); i < nchunks; i++)
                SX_CUDA(ctx, cudaEventSynchronize(r.done[int(i % kRingSlots)]));
        }
        return SXGPU_OK;
    };
    SX_TRY(finish(issue_all()));

    ctx->h2d_bytes += in_bytes;
    ctx->d2h_bytes += out_bytes;
    return SXGPU_OK;
}

// ---------------------------------------------------------------------------------------
// Batched blocks
// ---------------------------------------------------------------------------------------
static_assert(sizeof(sxgpu_block) == sizeof(BlockDesc), "descriptor layouts must match");

// Tile shape of the batched bulk kernel and of the bulk loopback: the large-block default.
constexpr int kBatchTile = 2048, kBatchStages = 4;
template <class Op> constexpr size_t batch_smem_bytes(bool local_scan)
{
    return size_t(kBatchStages) * (size_t(kBatchTile) * (Op::kSrcWords + Op::kDstWords) * 4 + 8 + sizeof(TileRecord)) +
           (local_scan ? (size_t(kBatchLocalBlocks) + 1) * sizeof(unsigned long long) : 0);
}
// Shapes of the bulk loopback kernel (three buffers per stage: 24 KiB per 1024 frames).
typedef void (*LoopKernel)(const BulkLoopbackArgs);
struct LoopShape {
    int tile, stages;
    LoopKernel kernel;
};
const LoopShape kLoopShapes[] = {
    {2048, 3, bulk_loopback_kernel<2048, 3>}, // default: 6 543 GB/s of 24 B/frame at 2^27 frames, against 6 085 for 4 stages
    {2048, 4, bulk_loopback_kernel<2048, 4>},
    {1024, 4, bulk_loopback_kernel<1024, 4>},
    {1024, 6, bulk_loopback_kernel<1024, 6>},
    {1024, 8, bulk_loopback_kernel<1024, 8>},
    {512, 8, bulk_loopback_kernel<512, 8>},
};
size_t loop_smem_bytes(const LoopShape &s)
{
    return 3 * size_t(s.stages) * s.tile * 8 + size_t(s.stages) * 8;
}

template <class Op>
int convert_batch(sxgpu_ctx *ctx, const sxgpu_block *blocks, uint32_t nblocks, int on_device,
                  size_t max_length, sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (nblocks == 0)
        return SXGPU_OK;
    if (!blocks)
        return ctx->invalid("null block list");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);

    const BlockDesc *d_blocks = reinterpret_cast<const BlockDesc *>(blocks);
    void *staged = nullptr;
    if (!on_device) {
        for (uint32_t i = 0; i < nblocks; i++) {
            if (blocks[i].length && (!blocks[i].src || !blocks[i].dest))
                return ctx->invalid("null sample buffer in block list");
            if (reinterpret_cast<uintptr_t>(blocks[i].src) % (Op::kSrcWords * 4) ||
                reinterpret_cast<uintptr_t>(blocks[i].dest) % (Op::kDstWords * 4))
                return ctx->invalid("batched blocks must be frame-aligned");
            max_length = std::max<size_t>(max_length, blocks[i].length);
        }
        // Stream-ordered staging: safe against back-to-back batches on any stream.  The
        // descriptors are followed by the exclusive prefix sum of their tile counts.
        SX_CUDA(ctx, cudaMallocFromPoolAsync(&staged, size_t(nblocks) * sizeof(BlockDesc) +
                                                          (size_t(nblocks) + 1) * sizeof(unsigned long long),
                                             ctx->scratch_pool, st));
    } else if (max_length == 0) {
        return ctx->invalid("max_length is required for device-resident block lists");
    }
    // From here on every return path gives the staging memory back.
    struct StagedGuard {
        void *p;
        cudaStream_t st;
        ~StagedGuard()
        {
            if (p)
                cudaFreeAsync(p, st);
        }
    } guard = {staged, st}, scan_guard = {nullptr, st};
    uint64_t host_tiles = 0;
    if (staged) {
        std::vector<unsigned long long> tile_start(size_t(nblocks) + 1);
        for (uint32_t i = 0; i < nblocks; i++) {
            tile_start[i] = host_tiles;
            host_tiles += (blocks[i].length + kBatchTile - 1) / kBatchTile;
        }
        tile_start[nblocks] = host_tiles;
        // (long lists only; short ones are summed by the kernel.)  Pageable source: copied before
        // cudaMemcpyAsync returns.
        if (nblocks > kBatchLocalBlocks)
            SX_CUDA(ctx, cudaMemcpyAsync(static_cast<char *>(staged) + size_t(nblocks) * sizeof(BlockDesc), tile_start.data(),
                                         tile_start.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
        // The caller may reuse `blocks` as soon as this call returns: when the list sits in pinned
        // memory cudaMemcpyAsync is truly asynchronous and would read it later, so the copy is
        // waited for here (a few microseconds for a list of this size; the kernels stay asynchronous).
        SX_CUDA(ctx, cudaMemcpyAsync(staged, blocks, size_t(nblocks) * sizeof(BlockDesc),
                                     cudaMemcpyHostToDevice, st));
        if (classify_pointer(ctx, blocks).pinned) {
            cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
            cudaStreamIsCapturing(st, &capturing);
            if (capturing == cudaStreamCaptureStatusNone)
                SX_CUDA(ctx, cudaStreamSynchronize(st));
        }
        d_blocks = static_cast<const BlockDesc *>(staged);
    }

    const int sms = ctx->prop.multiProcessorCount;
    // One chunk per CTA, CTAs in block-then-chunk order (batch_direct_kernel): the schedule of the
    // single-block default.  Every block gets the chunk count of the longest one and the CTAs past
    // a shorter block's end leave at once, so it is taken when that padding is small: host lists
    // are checked exactly; device-resident lists are taken at the caller's word (max_length) up to
    // a grid that bounds what a ragged list could waste.
    constexpr uint64_t kChunk = batch_direct_chunk<Op>();
    const uint64_t chunks_per_block = (uint64_t(max_length) + kChunk - 1) / kChunk;
    bool batch_direct = false;
    if (max_length > 4096 && (ctx->batch_variant == 0 || ctx->batch_variant == 2)) {
        const uint64_t grid = uint64_t(nblocks) * chunks_per_block;
        if (staged) {
            uint64_t used = 0;
            for (uint32_t i = 0; i < nblocks; i++)
                used += (blocks[i].length + kChunk - 1) / kChunk;
            batch_direct = grid <= 0x7fffffffu && (ctx->batch_variant == 2 || used * 4 >= grid * 3);
        } else {
            batch_direct = grid <= (ctx->batch_variant == 2 ? 0x7fffffffu : (uint64_t(1) << 21));
        }
    }
    if (max_length <= 4096) {
        // One warp per block: a 256-frame period is 128 x 16 bytes = 4 accesses per lane.
        int block = 256, warps = block / 32;
        uint64_t ctas = (uint64_t(nblocks) + warps - 1) / warps;
        int grid = ctx->warp_ctas_per_sm <= 0 ? int(std::min<uint64_t>(ctas, 0x7fffffffu))
                                              : int(std::min<uint64_t>(ctas, uint64_t(sms) * uint64_t(ctx->warp_ctas_per_sm)));
        batch_warp_kernel<Op><<<grid, block, 0, st>>>(d_blocks, nblocks);
    } else if (batch_direct) {
        batch_direct_kernel<Op><<<unsigned(uint64_t(nblocks) * chunks_per_block), 256, 0, st>>>(d_blocks, nblocks,
                                                                                            uint32_t(chunks_per_block));
    } else if (ctx->batch_variant == 1) {
        int block = 256;
        uint64_t slices = (max_length + 16383) / 16384; // ~128 KiB of frames per CTA pass
        uint64_t want = uint64_t(sms) * 8;
        uint32_t gy = uint32_t(std::max<uint64_t>(1, std::min<uint64_t>(slices, (want + nblocks - 1) / nblocks)));
        uint32_t gx = uint32_t(std::min<uint64_t>(nblocks, std::max<uint64_t>(1, want / gy)));
        batch_slice_kernel<Op><<<dim3(gx, gy), block, 0, st>>>(d_blocks, nblocks);
    } else {
        // Mid-size and large blocks: every block cut into tiles, all tiles of all blocks walked by
        // one persistent CTA per SM on the bulk-async schedule (bulk_batch_kernel).
        constexpr int TILE = kBatchTile;
        const int sm_grid_hint = sms; // the kernel finds the tile total itself; never more CTAs than SMs x occupancy
        if (nblocks <= kBatchLocalBlocks) {
            // Short lists: every CTA sums the tile counts itself.  One launch, no scratch.
            BatchBulkArgs a = {d_blocks, nullptr, nblocks, int(ctx->bulk_load_policy), int(ctx->bulk_store_policy)};
            auto k = bulk_batch_kernel<Op, TILE, kBatchStages, true>;
            const size_t smem = batch_smem_bytes<Op>(true);
            const uint64_t hint = staged ? std::max<uint64_t>(host_tiles, 1) : uint64_t(sm_grid_hint);
            k<<<persistent_grid(ctx, k, 256, smem, hint), 256, smem, st>>>(a);
        } else {
            unsigned long long *d_tile_start = nullptr;
            uint64_t hint = uint64_t(sm_grid_hint);
            if (staged) {
                d_tile_start = reinterpret_cast<unsigned long long *>(static_cast<char *>(staged) +
                                                                      size_t(nblocks) * sizeof(BlockDesc));
                hint = std::max<uint64_t>(host_tiles, 1);
            } else {
                SX_CUDA(ctx, cudaMallocFromPoolAsync(reinterpret_cast<void **>(&d_tile_start),
                                                     (size_t(nblocks) + 1) * sizeof(unsigned long long), ctx->scratch_pool, st));
                scan_guard.p = d_tile_start;
                batch_tile_scan_kernel<TILE><<<1, 1024, 0, st>>>(d_blocks, nblocks, d_tile_start);
                SX_CUDA(ctx, cudaGetLastError());
                ctx->launches++;
            }
            BatchBulkArgs a = {d_blocks, d_tile_start, nblocks, int(ctx->bulk_load_policy), int(ctx->bulk_store_policy)};
            auto k = bulk_batch_kernel<Op, TILE, kBatchStages, false>;
            const size_t smem = batch_smem_bytes<Op>(false);
            k<<<persistent_grid(ctx, k, 256, smem, hint), 256, smem, st>>>(a);
        }
    }
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

int64_t *option_slot(sxgpu_ctx *ctx, const char *key)
{
    struct {
        const char *name;
        int64_t *slot;
    } table[] = {
        {"rx_variant", &ctx->rx_variant},
        {"tx_variant", &ctx->tx_variant},
        {"unroll", &ctx->unroll},
        {"block", &ctx->block},
        {"ctas_per_sm", &ctx->ctas_per_sm},
        {"bulk_tile", &ctx->bulk_tile},
        {"bulk_stages", &ctx->bulk_stages},
        {"bulk_load_policy", &ctx->bulk_load_policy},
        {"bulk_store_policy", &ctx->bulk_store_policy},
        {"bulk_contiguous", &ctx->bulk_contiguous},
        {"host_chunk_frames", &ctx->host_chunk_frames},
        {"host_chunk_min_frames", &ctx->host_chunk_min_frames},
        {"host_mode", &ctx->host_mode},
        {"small_mode", &ctx->small_mode},
        {"host_in_mode", &ctx->host_in_mode},
        {"host_out_mode", &ctx->host_out_mode},
        {"bounce_nt", &ctx->bounce_nt},
        {"pipeline_mode", &ctx->pipeline_mode},
        {"zero_copy_max_frames", &ctx->zero_copy_max_frames},
        {"resident_max_frames", &ctx->resident_max_frames},
        {"zero_copy_variant", &ctx->zero_copy_variant},
        {"bank_repeat_variant", &ctx->bank_repeat_variant},
        {"bank_split_variant", &ctx->bank_split_variant},
        {"warp_ctas_per_sm", &ctx->warp_ctas_per_sm},
        {"batch_variant", &ctx->batch_variant},
        {"loopback_variant", &ctx->loopback_variant},
        {"bounce_threads", &ctx->bounce_threads},
        {"numa_local_alloc", &ctx->numa_local_alloc},
        {"numa_node", &ctx->numa_node},
    };
    for (auto &e : table)
        if (std::strcmp(e.name, key) == 0)
            return e.slot;
    return nullptr;
}

template <class Op> int prepare_bulk_kernels(sxgpu_ctx *ctx)
{
    const BulkShape shapes[] = {{4096, 3}, {3072, 4}, {2048, 6}, {2048, 5}, {2048, 4},
                                {2048, 3}, {1024, 6}, {1024, 4}, {512, 4}};
    for (BulkShape s : shapes) {
        SX_CUDA(ctx, cudaFuncSetAttribute(bulk_kernel<Op>(s),
                                          cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          int(bulk_smem_bytes<Op>(s))));
        if (BulkKernel skewed = bulk_skew_kernel<Op>(s))
            SX_CUDA(ctx, cudaFuncSetAttribute(skewed, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              int(bulk_smem_bytes<Op>(s, true))));
    }
    return SXGPU_OK;
}

} // namespace

// ---------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------
extern "C" {

int sxgpu_abi_version(void) { return SXGPU_ABI_VERSION; }

const char *sxgpu_strerror(int code)
{
    switch (code) {
    case SXGPU_OK: return "ok";
    case SXGPU_ERR_INVALID: return "invalid argument";
    case SXGPU_ERR_CUDA: return "CUDA error";
    case SXGPU_ERR_NO_DEVICE: return "no usable sm_100 device";
    case SXGPU_ERR_NOMEM: return "out of memory";
    case SXGPU_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown error";
    }
}

const char *sxgpu_last_error(sxgpu_ctx *ctx)
{
    // The message is copied into storage of the calling thread, so the pointer stays valid (and
    // its contents unchanged) until this thread asks again, whatever other threads do meanwhile.
    static thread_local std::string mine;
    if (!ctx)
        return "";
    std::lock_guard<std::mutex> lock(ctx->err_mutex);
    mine = ctx->last_error;
    return mine.c_str();
}

int sxgpu_init(int device, sxgpu_ctx **out)
{
    if (!out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        cudaGetLastError();
        return SXGPU_ERR_NO_DEVICE;
    }
    sxgpu_ctx *ctx = new sxgpu_ctx();
    ctx->device = device;
    auto bail = [&](int code) {
        if (ctx->scratch_pool) cudaMemPoolDestroy(ctx->scratch_pool);
        if (ctx->d_stats) cudaFree(ctx->d_stats);
        if (ctx->h_stats) cudaFreeHost(ctx->h_stats);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        cudaGetLastError();
        delete ctx;
        return code;
    };
    if (cudaGetDeviceProperties(&ctx->prop, device) != cudaSuccess)
        return bail(SXGPU_ERR_NO_DEVICE);
    // The library carries sm_100a code only (no PTX, no other architectures).
    if (ctx->prop.major != 10)
        return bail(SXGPU_ERR_NO_DEVICE);
    if (cudaSetDevice(device) != cudaSuccess)
        return bail(SXGPU_ERR_CUDA);
    // An ordinary (blocking) stream: it orders with the legacy default stream exactly like any
    // cudaStreamCreate() stream, so a caller that fills a buffer on the default stream and then
    // converts it on "the context's stream" (or reads the result back) needs no extra sync.
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamDefault) != cudaSuccess)
        return bail(SXGPU_ERR_CUDA);
    read_gpu_locality(ctx);
    if (cudaMalloc(&ctx->d_stats, sizeof(StatsAcc)) != cudaSuccess ||
        cudaHostAlloc(&ctx->h_stats, sizeof(StatsAcc), cudaHostAllocDefault) != cudaSuccess)
        return bail(SXGPU_ERR_NOMEM);
    if (prepare_bulk_kernels<RxCf32>(ctx) != SXGPU_OK || prepare_bulk_kernels<TxCf32>(ctx) != SXGPU_OK ||
        prepare_bulk_kernels<RxCs16>(ctx) != SXGPU_OK || prepare_bulk_kernels<TxCs16>(ctx) != SXGPU_OK ||
        prepare_bulk_kernels<RxS16Cf32>(ctx) != SXGPU_OK || prepare_bulk_kernels<TxCf32S16>(ctx) != SXGPU_OK)
        return bail(SXGPU_ERR_CUDA);
    if (cudaFuncSetAttribute(bulk_batch_kernel<RxCf32, kBatchTile, kBatchStages, false>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, int(batch_smem_bytes<RxCf32>(false))) != cudaSuccess ||
        cudaFuncSetAttribute(bulk_batch_kernel<TxCf32, kBatchTile, kBatchStages, false>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, int(batch_smem_bytes<TxCf32>(false))) != cudaSuccess ||
        cudaFuncSetAttribute(bulk_batch_kernel<RxCf32, kBatchTile, kBatchStages, true>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, int(batch_smem_bytes<RxCf32>(true))) != cudaSuccess ||
        cudaFuncSetAttribute(bulk_batch_kernel<TxCf32, kBatchTile, kBatchStages, true>,
                             cudaFuncAttributeMaxDynamicSharedMemorySize, int(batch_smem_bytes<TxCf32>(true))) != cudaSuccess)
        return bail(SXGPU_ERR_CUDA);
    {
        // Stream-ordered scratch (descriptor lists staged from the host, tile counts of long lists)
        // comes from a pool of the context's own that keeps what it is given back: the default
        // pool returns memory to the system at every synchronisation, and the next batch then
        // paid a fresh allocation -- several hundred microseconds, twice the conversion itself.
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&ctx->scratch_pool, &props) != cudaSuccess)
            return bail(SXGPU_ERR_CUDA);
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(ctx->scratch_pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    for (const LoopShape &shape : kLoopShapes)
        if (cudaFuncSetAttribute(shape.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 int(loop_smem_bytes(shape))) != cudaSuccess)
            return bail(SXGPU_ERR_CUDA);
    *out = ctx;
    return SXGPU_OK;
}

int sxgpu_destroy(sxgpu_ctx *ctx)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (ctx->live_banks.load() != 0)
        return ctx->invalid("destroy the context's stream banks first");
    if (ctx->live_dsp.load() != 0)
        return ctx->invalid("destroy the context's filters, oscillators and channelizers first");
    quiesce(ctx);
    for (HostLane &lane : ctx->lanes) {
        HostRing &r = lane.ring;
        for (int i = 0; i < kRingSlots; i++) {
            if (r.d_in[i]) cudaFree(r.d_in[i]);
            if (r.d_out[i]) cudaFree(r.d_out[i]);
            if (r.h_in[i]) cudaFreeHost(r.h_in[i]);
            if (r.h_out[i]) cudaFreeHost(r.h_out[i]);
            if (r.events) {
                cudaEventDestroy(r.copied_in[i]);
                cudaEventDestroy(r.converted[i]);
                cudaEventDestroy(r.done[i]);
            }
        }
        if (lane.s_h2d) cudaStreamDestroy(lane.s_h2d);
        if (lane.s_comp) cudaStreamDestroy(lane.s_comp);
        if (lane.s_d2h) cudaStreamDestroy(lane.s_d2h);
        for (int i = 0; i < kRingSlots; i++)
            if (lane.s_slot[i]) cudaStreamDestroy(lane.s_slot[i]);
        if (lane.s_resident) cudaStreamDestroy(lane.s_resident); // its kernel has left: asked to, and the device was synchronised
        if (lane.mailbox) cudaFreeHost(lane.mailbox);
        if (lane.flag) cudaFreeHost(lane.flag);
        if (lane.d_arrivals) cudaFree(lane.d_arrivals);
    }
    if (ctx->scratch_pool) cudaMemPoolDestroy(ctx->scratch_pool);
    if (ctx->d_stats) cudaFree(ctx->d_stats);
    if (ctx->h_stats) cudaFreeHost(ctx->h_stats);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return SXGPU_OK;
}

int sxgpu_device_info(sxgpu_ctx *ctx, sxgpu_info *out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    std::memset(out, 0, sizeof *out);
    out->device = ctx->device;
    out->sm_count = ctx->prop.multiProcessorCount;
    out->cc_major = ctx->prop.major;
    out->cc_minor = ctx->prop.minor;
    out->l2_bytes = uint64_t(ctx->prop.l2CacheSize);
    out->hbm_bytes = uint64_t(ctx->prop.totalGlobalMem);
    std::snprintf(out->name, sizeof out->name, "%.63s", ctx->prop.name);
    return SXGPU_OK;
}

int sxgpu_convert_rx_buffer(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                            size_t dest_offset, size_t length, sxgpu_stream stream)
{
    int r = convert_entry<RxCf32>(ctx, d_src, src_offset, d_dest, dest_offset, length, 0.0f,
                                  ctx ? ctx->rx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_tx_buffer(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                            size_t dest_offset, size_t length, float tx_threshold2,
                            sxgpu_stream stream)
{
    int r = convert_entry<TxCf32>(ctx, d_src, src_offset, d_dest, dest_offset, length,
                                  tx_threshold2, ctx ? ctx->tx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_convert_rx_buffer_cs16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset,
                                 void *d_dest, size_t dest_offset, size_t length,
                                 sxgpu_stream stream)
{
    int r = convert_entry<RxCs16>(ctx, d_src, src_offset, d_dest, dest_offset, length, 0.0f,
                                  ctx ? ctx->rx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_tx_buffer_cs16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset,
                                 void *d_dest, size_t dest_offset, size_t length,
                                 float tx_threshold2, sxgpu_stream stream)
{
    int r = convert_entry<TxCs16>(ctx, d_src, src_offset, d_dest, dest_offset, length,
                                  tx_threshold2, ctx ? ctx->tx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_convert_rx_buffer_s16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                                size_t dest_offset, size_t length, sxgpu_stream stream)
{
    int r = convert_entry<RxS16Cf32>(ctx, d_src, src_offset, d_dest, dest_offset, length, 0.0f,
                                     ctx ? ctx->rx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_tx_buffer_s16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                                size_t dest_offset, size_t length, float tx_threshold2,
                                sxgpu_stream stream)
{
    int r = convert_entry<TxCf32S16>(ctx, d_src, src_offset, d_dest, dest_offset, length,
                                     tx_threshold2, ctx ? ctx->tx_variant : 0, stream);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_convert_rx_batch(sxgpu_ctx *ctx, const sxgpu_block *blocks, uint32_t nblocks,
                           int blocks_on_device, size_t max_length, sxgpu_stream stream)
{
    return convert_batch<RxCf32>(ctx, blocks, nblocks, blocks_on_device, max_length, stream);
}

int sxgpu_convert_tx_batch(sxgpu_ctx *ctx, const sxgpu_block *blocks, uint32_t nblocks,
                           int blocks_on_device, size_t max_length, sxgpu_stream stream)
{
    return convert_batch<TxCf32>(ctx, blocks, nblocks, blocks_on_device, max_length, stream);
}

int sxgpu_convert_loopback(sxgpu_ctx *ctx, const void *d_i2s_in, void *d_cf32, void *d_i2s_out,
                           size_t length, float tx_threshold2, sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (length == 0)
        return SXGPU_OK;
    if (!d_i2s_in || !d_i2s_out)
        return ctx->invalid("null sample buffer");
    auto misaligned = [](const void *p) { return reinterpret_cast<uintptr_t>(p) % 16 != 0; };
    if (misaligned(d_i2s_in) || misaligned(d_i2s_out) || (d_cf32 && misaligned(d_cf32)))
        return ctx->invalid("loopback buffers must be 16-byte aligned");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    if (ctx->loopback_variant == 0 || ctx->loopback_variant == 2) {
        // One tile per CTA, handed out in index order by the hardware (see launch_convert): two
        // 16-byte vectors per thread in flight, 6.8 TB/s of 24 B/frame at 2^27 frames.
        LoopbackArgs a = {static_cast<const char *>(d_i2s_in), static_cast<char *>(d_cf32),
                          static_cast<char *>(d_i2s_out), length / 2, length, tx_threshold2};
        constexpr int block = 256, U = 2;
        uint64_t tiles = std::max<uint64_t>(1, (a.nvec + uint64_t(block) * U - 1) / (uint64_t(block) * U));
        loopback_kernel<U><<<unsigned(std::min<uint64_t>(tiles, 0x7fffffffu)), block, 0, st>>>(a);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    } else if (ctx->loopback_variant == 3 && length >= 2) {
        // Bulk-async schedule over the even part; an odd last frame goes through the vector kernel.
        const uint64_t even = uint64_t(length) & ~uint64_t(1);
        BulkLoopbackArgs b = {static_cast<const char *>(d_i2s_in), static_cast<char *>(d_cf32),
                              static_cast<char *>(d_i2s_out), even, tx_threshold2, int(ctx->bulk_load_policy),
                              int(ctx->bulk_store_policy)};
        const LoopShape *shape = &kLoopShapes[0];
        if (ctx->bulk_tile || ctx->bulk_stages) { // tuning: option bulk_tile / bulk_stages select a shape
            shape = nullptr;
            for (const LoopShape &c : kLoopShapes)
                if (c.tile == (ctx->bulk_tile ? ctx->bulk_tile : 2048) && c.stages == (ctx->bulk_stages ? ctx->bulk_stages : 3))
                    shape = &c;
            if (!shape)
                return ctx->invalid("unsupported bulk_tile/bulk_stages combination for the loopback");
        }
        const uint64_t ntiles = (even + shape->tile - 1) / shape->tile;
        const size_t smem = loop_smem_bytes(*shape);
        shape->kernel<<<persistent_grid(ctx, shape->kernel, 256, smem, ntiles), 256, smem, st>>>(b);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
        if (length & 1) {
            const size_t off = even * 8;
            LoopbackArgs t = {static_cast<const char *>(d_i2s_in) + off, d_cf32 ? static_cast<char *>(d_cf32) + off : nullptr,
                              static_cast<char *>(d_i2s_out) + off, 0, 1, tx_threshold2};
            loopback_kernel<4><<<1, 32, 0, st>>>(t);
            SX_CUDA(ctx, cudaGetLastError());
            ctx->launches++;
        }
    } else {
        LoopbackArgs a = {static_cast<const char *>(d_i2s_in), static_cast<char *>(d_cf32),
                          static_cast<char *>(d_i2s_out), length / 2, length, tx_threshold2};
        int block = int(ctx->block ? ctx->block : 256);
        constexpr int U = 4;
        uint64_t tiles = (a.nvec + uint64_t(block) * U - 1) / (uint64_t(block) * U);
        int grid = persistent_grid(ctx, loopback_kernel<U>, block, 0, tiles);
        loopback_kernel<U><<<grid, block, 0, st>>>(a);
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
    }
    ctx->frames_rx += length;
    ctx->frames_tx += length;
    return SXGPU_OK;
}

// ---- stream bank ------------------------------------------------------------------------
} // extern "C"

struct sxgpu_bank {
    sxgpu_ctx *ctx = nullptr;
    BankState st = {};
    void *arena = nullptr; // one allocation for every per-stream array
    bool external_capture = false; // capture slots are filled by sxgpu_bank_ingest, not synthesised
};

namespace {

template <class T> T *carve(char *&cursor, size_t count)
{
    uintptr_t p = (reinterpret_cast<uintptr_t>(cursor) + 255) & ~uintptr_t(255);
    cursor = reinterpret_cast<char *>(p) + count * sizeof(T);
    return reinterpret_cast<T *>(p);
}

// Measured (profiles/r01_summary.md section 6): up to a few thousand streams an iteration is
// launch-bound and planning inside the data kernels saves two launches; at 65536 streams the
// separate thread-per-stream plan kernels are 20 % faster.
constexpr uint32_t kBankFusedPlanStreams = 8192;


int per_stream_grid(uint32_t nstreams, int block)
{
    return int((nstreams + block - 1) / block);
}

int per_warp_grid(const sxgpu_ctx *ctx, uint32_t nstreams, int block)
{
    uint64_t ctas = (uint64_t(nstreams) + block / 32 - 1) / (block / 32);
    if (ctx->warp_ctas_per_sm <= 0) // one CTA per eight streams, handed out in order by the hardware
        return int(std::min<uint64_t>(ctas, 0x7fffffffu));
    return int(std::min<uint64_t>(ctas, uint64_t(ctx->prop.multiProcessorCount) * uint64_t(ctx->warp_ctas_per_sm)));
}

// The separate read / write calls of a large bank go through the plan + data kernels too
// (option bank_split_variant: 0 auto, 1 = always the warp-per-stream kernels).
bool bank_split_direct(const sxgpu_ctx *ctx, const BankState &b, const void *d_cf32)
{
    return ctx->bank_split_variant != 1 && bank_is_large(b) && reinterpret_cast<uintptr_t>(d_cf32) % 16 == 0;
}

template <class T>
int copy_out(sxgpu_bank *bank, T *h_dst, const void *d_src, cudaStream_t st)
{
    if (!h_dst)
        return SXGPU_OK;
    SX_CUDA(bank->ctx, cudaMemcpyAsync(h_dst, d_src, size_t(bank->st.nstreams) * sizeof(T),
                                       cudaMemcpyDeviceToHost, st));
    return SXGPU_OK;
}

} // namespace

extern "C" {

int sxgpu_bank_create(sxgpu_ctx *ctx, const sxgpu_bank_config *config, sxgpu_bank **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (!config || config->nstreams == 0)
        return ctx->invalid("a bank needs at least one stream");
    if (!(config->sample_rate >= 1.0))
        return ctx->invalid("sample rate must be at least 1 Hz");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));

    sxplan::Geometry geo = sxplan::geometry_for_period(config->period);
    const size_t n = config->nstreams;
    sxgpu_bank *bank = new sxgpu_bank();
    bank->ctx = ctx;
    BankState &b = bank->st;
    b.nstreams = config->nstreams;
    b.period = uint32_t(geo.period);
    b.ring = geo.buffer;
    b.sample_rate = config->sample_rate;
    b.thr2 = config->tx_threshold2;
    b.seed = config->seed;

    size_t bytes = 0;
    bytes += 3 * (n * sizeof(long long) + 256);                       // clock, rx/tx position
    bytes += 3 * (n * sizeof(int) + 256) + (n * sizeof(long long) + 256); // results
    bytes += 5 * (n * sizeof(long long) + 256) + (n * sizeof(BlockDesc) + 256); // plans
    bytes += n * geo.period * 8 + 256;                                // capture staging
    bytes += n * geo.buffer * 8 + 256;                                // playback rings
    cudaError_t e = cudaMalloc(&bank->arena, bytes);
    if (e != cudaSuccess) {
        delete bank;
        return ctx->fail(e, "cudaMalloc(stream bank)");
    }
    // Zero everything: counters start at 0 and an untouched ring is silence.
    e = cudaMemsetAsync(bank->arena, 0, bytes, ctx->stream);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cudaFree(bank->arena);
        delete bank;
        return ctx->fail(e, "cudaMemset(stream bank)");
    }
    char *cur = static_cast<char *>(bank->arena);
    b.clock = carve<long long>(cur, n);
    b.rx_position = carve<long long>(cur, n);
    b.tx_position = carve<long long>(cur, n);
    b.rx_ret = carve<int>(cur, n);
    b.rx_flags = carve<int>(cur, n);
    b.tx_ret = carve<int>(cur, n);
    b.rx_time_ns = carve<long long>(cur, n);
    b.rx_first_frame = carve<long long>(cur, n);
    b.tx_write_position = carve<long long>(cur, n);
    b.tx_gap_start = carve<long long>(cur, n);
    b.tx_gap_length = carve<long long>(cur, n);
    b.tx_ring_offset = carve<long long>(cur, n);
    b.rx_blocks = carve<BlockDesc>(cur, n);
    b.capture_stage = carve<char>(cur, n * geo.period * 8);
    b.playback_ring = carve<char>(cur, n * geo.buffer * 8);
    ctx->live_banks++;
    *out = bank;
    return SXGPU_OK;
}

int sxgpu_bank_destroy(sxgpu_bank *bank)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    quiesce(bank->ctx);
    cudaFree(bank->arena);
    bank->ctx->live_banks--;
    delete bank;
    return SXGPU_OK;
}

int sxgpu_bank_ring_frames(sxgpu_bank *bank, uint64_t *ring_frames)
{
    if (!bank || !ring_frames)
        return SXGPU_ERR_INVALID;
    *ring_frames = bank->st.ring;
    return SXGPU_OK;
}

int sxgpu_bank_advance(sxgpu_bank *bank, int64_t frames, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (frames < 0)
        return ctx->invalid("the sample clock only runs forward");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    bank_advance_kernel<<<per_stream_grid(bank->st.nstreams, 256), 256, 0, call_stream(bank->ctx, stream)>>>(
        bank->st, frames);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

int sxgpu_bank_read(sxgpu_bank *bank, void *d_cf32, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("CF32 buffer must be 8-byte aligned device memory");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    const BankState &b = bank->st;
    if (bank_split_direct(ctx, b, d_cf32)) {
        // large banks: decisions by a thread per stream, then capture and RX conversion by CTAs that
        // take one chunk each (sx_bank.cuh, bank_repeat_data_kernel in read mode)
        SX_CUDA(ctx, (launch_bank_planned<kBankModeRead, 4>(b, static_cast<char *>(d_cf32), bank->external_capture, 0, nullptr, 0,
                                                            st, IdentityHook())));
        ctx->launches += 2;
        ctx->frames_rx += uint64_t(b.nstreams) * b.period;
        return SXGPU_OK;
    }
    const bool fused = b.nstreams <= kBankFusedPlanStreams;
    if (!fused)
        bank_plan_read_kernel<<<per_stream_grid(b.nstreams, 256), 256, 0, st>>>(b, static_cast<char *>(d_cf32));
    bank_capture_kernel<<<per_warp_grid(ctx, b.nstreams, 256), 256, 0, st>>>(b, static_cast<char *>(d_cf32), fused,
                                                                             !bank->external_capture);
    batch_warp_kernel<RxCf32><<<per_warp_grid(ctx, b.nstreams, 256), 256, 0, st>>>(b.rx_blocks, b.nstreams);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches += fused ? 2 : 3;
    ctx->frames_rx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

int sxgpu_bank_write(sxgpu_bank *bank, const void *d_cf32, int flags, const long long *d_time_ns,
                     long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("CF32 buffer must be 8-byte aligned device memory");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    const BankState &b = bank->st;
    if (bank_split_direct(ctx, b, d_cf32)) {
        SX_CUDA(ctx, (launch_bank_planned<kBankModeWrite, 4>(b, const_cast<char *>(static_cast<const char *>(d_cf32)), false, flags,
                                                             d_time_ns, rx_time_offset_ns, st, IdentityHook())));
        ctx->launches += 2;
        ctx->frames_tx += uint64_t(b.nstreams) * b.period;
        return SXGPU_OK;
    }
    const bool fused = b.nstreams <= kBankFusedPlanStreams;
    if (!fused)
        bank_plan_write_kernel<<<per_stream_grid(b.nstreams, 256), 256, 0, st>>>(b, flags, d_time_ns,
                                                                             rx_time_offset_ns, false);
    bank_tx_kernel<<<per_warp_grid(ctx, b.nstreams, 256), 256, 0, st>>>(
        b, static_cast<const char *>(d_cf32), flags, d_time_ns, rx_time_offset_ns, fused);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches += fused ? 1 : 2;
    ctx->frames_tx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

int sxgpu_bank_repeat(sxgpu_bank *bank, void *d_cf32, long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("CF32 buffer must be 8-byte aligned device memory");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    const BankState &b = bank->st;
    char *cf = static_cast<char *>(d_cf32);
    const bool ext = bank->external_capture;
    auto warp_variant = [&](auto kernel, uint64_t k) {
        const uint64_t chunks = (uint64_t(b.nstreams) + k - 1) / k;
        kernel<<<persistent_grid(ctx, kernel, 256, 0, (chunks + 7) / 8), 256, 0, st>>>(b, cf, rx_time_offset_ns, ext,
                                                                                       IdentityHook());
    };
    // Schedules.  K streams per warp round: lanes 0..K-1 take K streams' decisions side by side, so
    // a larger K spends fewer issue slots on the timestamp arithmetic; a smaller K spreads few
    // streams over more warps.  1/2/4 and 100 (a CTA takes 32 streams per round, its first warp
    // decides for all of them) carry each stream through memory stage by stage (each stage reading
    // from L2 what the previous one wrote); 201/202/204 keep the stages' intermediates in registers
    // and only store.  Measured crossovers: profiles/r02_summary.md.
    const bool reg_ok = (b.period % 2 == 0) && reinterpret_cast<uintptr_t>(d_cf32) % 16 == 0;
    int64_t k = ctx->bank_repeat_variant;
    if (k == 0) {
        if (b.nstreams <= 2048)
            k = reg_ok ? 201 : 1;
        else if (!bank_is_large(b) || !reg_ok)
            k = b.nstreams <= 8192 ? 2 : b.nstreams <= 32768 ? 4 : 100;
        else
            k = ext ? 604 : 600; // decisions first, then the samples by hardware-scheduled CTAs
    }
    if (k >= 200 && !reg_ok)
        return ctx->invalid("the register schedules need an even period and a 16-byte aligned CF32 buffer");
    switch (k) {
    case 1: warp_variant(bank_repeat_warp_kernel<1>, 1); break;
    case 2: warp_variant(bank_repeat_warp_kernel<2>, 2); break;
    case 4: warp_variant(bank_repeat_warp_kernel<4>, 4); break;
    case 100: {
        const uint64_t groups = (uint64_t(b.nstreams) + kRepeatGroup - 1) / kRepeatGroup;
        bank_repeat_kernel<<<persistent_grid(ctx, bank_repeat_kernel, 256, 0, groups), 256, 0, st>>>(b, cf, rx_time_offset_ns, ext);
        break;
    }
    case 201: warp_variant(bank_repeat_warp_kernel<1, true>, 1); break;
    case 202: warp_variant(bank_repeat_warp_kernel<2, true>, 2); break;
    case 204: warp_variant(bank_repeat_warp_kernel<4, true>, 4); break;
    case 600:   // decisions by a thread-per-stream kernel, then the samples by hardware-scheduled CTAs (two vectors per thread)
    case 604: { // ... four vectors per thread
        if (b.period < 4)
            return ctx->invalid("the direct schedules need a period of at least four frames");
        SX_CUDA(ctx, (k == 600 ? launch_bank_planned<kBankModeRepeat, 2>(b, cf, ext, SX_HAS_TIME, nullptr, rx_time_offset_ns, st,
                                                                          IdentityHook())
                               : launch_bank_planned<kBankModeRepeat, 4>(b, cf, ext, SX_HAS_TIME, nullptr, rx_time_offset_ns, st,
                                                                          IdentityHook())));
        ctx->launches++;
        break;
    }
    default: return ctx->invalid("bank_repeat_variant must be 0 (auto), 1, 2, 4, 100, 201, 202, 204, 600 or 604");
    }
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches += 1;
    ctx->frames_rx += uint64_t(b.nstreams) * b.period;
    ctx->frames_tx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

// The repeater iteration split around a kernel of the caller's: begin = the read, with the
// CF32 block marked persisting in L2 for the stream; end = the timed write of that block, after
// which the mark is lifted.  In between the caller launches whatever it likes on the same stream.
int sxgpu_bank_repeat_begin(sxgpu_bank *bank, void *d_cf32, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (!d_cf32)
        return ctx->invalid("null CF32 buffer");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    const size_t bytes = size_t(bank->st.nstreams) * bank->st.period * 8;
    const size_t window = std::min<size_t>(bytes, size_t(ctx->prop.accessPolicyMaxWindowSize));
    if (window > 0 && ctx->prop.persistingL2CacheMaxSize > 0) {
        if (!ctx->l2_carveout_set) { // once: let up to three quarters of L2 hold persisting lines
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize,
                               std::min<size_t>(size_t(ctx->prop.persistingL2CacheMaxSize), size_t(ctx->prop.l2CacheSize) / 4 * 3));
            cudaGetLastError();
            ctx->l2_carveout_set = true;
        }
        cudaStreamAttrValue attr = {};
        attr.accessPolicyWindow.base_ptr = d_cf32;
        attr.accessPolicyWindow.num_bytes = window;
        attr.accessPolicyWindow.hitRatio = 1.0f;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
        if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess)
            cudaGetLastError(); // a hint only: the iteration is correct without it
    }
    return sxgpu_bank_read(bank, d_cf32, stream);
}

int sxgpu_bank_repeat_end(sxgpu_bank *bank, const void *d_cf32, long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    int rc = sxgpu_bank_write(bank, d_cf32, SX_HAS_TIME, nullptr, rx_time_offset_ns, stream);
    cudaStreamAttrValue attr = {};
    attr.accessPolicyWindow.num_bytes = 0; // lift the window for whatever the stream does next
    if (cudaStreamSetAttribute(call_stream(bank->ctx, stream), cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess)
        cudaGetLastError();
    return rc;
}

int sxgpu_bank_ingest(sxgpu_bank *bank, uint32_t first_stream, uint32_t nstreams, const void *i2s,
                      sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    const BankState &b = bank->st;
    if (nstreams == 0) {
        bank->external_capture = true;
        return SXGPU_OK;
    }
    if (!i2s || uint64_t(first_stream) + nstreams > b.nstreams)
        return ctx->invalid("ingest range outside the bank");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    // The capture slots of consecutive streams are contiguous: one copy, from wherever the frames
    // are (pinned or pageable host memory, or device memory).
    SX_CUDA(ctx, cudaMemcpyAsync(b.capture_stage + size_t(first_stream) * b.period * 8, i2s,
                                 size_t(nstreams) * b.period * 8, cudaMemcpyDefault, call_stream(bank->ctx, stream)));
    if (!classify_pointer(ctx, i2s).on_device)
        ctx->h2d_bytes += uint64_t(nstreams) * b.period * 8;
    bank->external_capture = true;
    return SXGPU_OK;
}

int sxgpu_bank_drain(sxgpu_bank *bank, uint32_t first_stream, uint32_t nstreams, size_t nframes, void *i2s,
                     sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    const BankState &b = bank->st;
    if (nstreams == 0 || nframes == 0)
        return SXGPU_OK;
    if (!i2s || uint64_t(first_stream) + nstreams > b.nstreams || nframes > b.ring)
        return ctx->invalid("drain range outside the bank or longer than a ring");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    HostPtrInfo di = classify_pointer(ctx, i2s);
    if (!di.device_alias || di.foreign_device || reinterpret_cast<uintptr_t>(di.device_alias) % 8)
        return ctx->invalid("drain destination must be device memory or pinned host memory, 8-byte aligned");
    bank_drain_kernel<<<per_warp_grid(ctx, nstreams, 256), 256, 0, call_stream(bank->ctx, stream)>>>(
        b, first_stream, nstreams, uint32_t(nframes), static_cast<char *>(di.device_alias));
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    if (!di.on_device)
        ctx->d2h_bytes += uint64_t(nstreams) * nframes * 8;
    return SXGPU_OK;
}

int sxgpu_bank_device_view(sxgpu_bank *bank, void *out, size_t out_bytes, int *external_capture)
{
    if (!bank || !out)
        return SXGPU_ERR_INVALID;
    if (out_bytes != sizeof(BankState))
        return bank->ctx->invalid("sxgpu_bank_device_view: size mismatch (header and library disagree)");
    std::memcpy(out, &bank->st, sizeof(BankState));
    if (external_capture)
        *external_capture = bank->external_capture ? 1 : 0;
    return SXGPU_OK;
}

int sxgpu_bank_last_read(sxgpu_bank *bank, int32_t *h_ret, int32_t *h_flags, int64_t *h_time_ns,
                         sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    SX_TRY(copy_out(bank, h_ret, bank->st.rx_ret, st));
    SX_TRY(copy_out(bank, h_flags, bank->st.rx_flags, st));
    SX_TRY(copy_out(bank, reinterpret_cast<long long *>(h_time_ns), bank->st.rx_time_ns, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int sxgpu_bank_last_write(sxgpu_bank *bank, int32_t *h_ret, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    SX_TRY(copy_out(bank, h_ret, bank->st.tx_ret, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int sxgpu_bank_positions(sxgpu_bank *bank, int64_t *h_clock, int64_t *h_rx_position,
                         int64_t *h_tx_position, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    SX_TRY(copy_out(bank, reinterpret_cast<long long *>(h_clock), bank->st.clock, st));
    SX_TRY(copy_out(bank, reinterpret_cast<long long *>(h_rx_position), bank->st.rx_position, st));
    SX_TRY(copy_out(bank, reinterpret_cast<long long *>(h_tx_position), bank->st.tx_position, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int sxgpu_bank_playback(sxgpu_bank *bank, uint32_t index, int64_t position, size_t nframes,
                        void *h_i2s, sxgpu_stream stream)
{
    if (!bank || !h_i2s)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    const BankState &b = bank->st;
    if (index >= b.nstreams || position < 0 || nframes > b.ring)
        return ctx->invalid("playback window outside the stream's ring");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(bank->ctx, stream);
    if (nframes == 0)
        return SXGPU_OK;
    // The rings are stored time-major (sx_bank.cuh, ring_frame): gather the window on the device,
    // then one copy out.
    void *tmp = nullptr;
    SX_CUDA(ctx, cudaMallocAsync(&tmp, nframes * 8, st));
    const int grid = int(std::min<uint64_t>((nframes + 255) / 256, uint64_t(ctx->prop.multiProcessorCount) * 4));
    bank_gather_kernel<<<grid, 256, 0, st>>>(b, index, position, nframes, static_cast<char *>(tmp));
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(h_i2s, tmp, nframes * 8, cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(tmp, st);
    if (e != cudaSuccess)
        return ctx->fail(e, "sxgpu_bank_playback");
    ctx->launches++;
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

// ---- stateful IIR filters (sx_iir.cuh) --------------------------------------------------------
} // extern "C"

struct sxgpu_iir {
    sxgpu_ctx *ctx = nullptr;
    IirView view = {};      // the state in device memory and the float32 coefficients
    DevPtr<float> state;    // view.state
    DevPtr<double> powers;  // sxgpu_iir_apply_long's P_j = A^(2^j) (sx_iir.cuh), in device memory
};

namespace {

// P_0 .. P_kIirPowers-1 of sx_iir.cuh's carry, [j][kIirDim][kIirDim] with zeros outside the
// 2S x 2S corner: A column by column (one float64 step of the cascade on zero input from a unit
// state), then repeated squaring, each entry summed left to right.  The build's -ffp-contract=off
// keeps every operation one rounding, as on the device and in tests/sxiir_long.py.
std::vector<double> iir_power_chain(const IirCoeffs &k)
{
    const int n = 2 * int(k.nsections);
    constexpr size_t kMat = size_t(kIirDim) * kIirDim;
    std::vector<double> p(kIirPowers * kMat, 0.0);
    for (int col = 0; col < n; col++) {
        double z[kIirDim] = {};
        z[col] = 1.0;
        double x = 0.0;
        for (int q = 0; q < int(k.nsections); q++) {
            const double b0 = k.b0[q], b1 = k.b1[q], b2 = k.b2[q], a1 = k.a1[q], a2 = k.a2[q];
            const double y = b0 * x + z[2 * q];
            const double z0 = (b1 * x - a1 * y) + z[2 * q + 1];
            const double z1 = b2 * x - a2 * y;
            z[2 * q] = z0;
            z[2 * q + 1] = z1;
            x = y;
        }
        for (int i = 0; i < n; i++)
            p[size_t(i) * kIirDim + col] = z[i];
    }
    for (int j = 1; j < kIirPowers; j++) {
        const double *a = &p[(j - 1) * kMat];
        double *out = &p[j * kMat];
        for (int i = 0; i < n; i++)
            for (int col = 0; col < n; col++) {
                double acc = a[size_t(i) * kIirDim] * a[col];
                for (int m = 1; m < n; m++)
                    acc = acc + a[size_t(i) * kIirDim + m] * a[size_t(m) * kIirDim + col];
                out[size_t(i) * kIirDim + col] = acc;
            }
    }
    return p;
}

// sxgpu_iir_apply_long's chunk length: a function of the shape alone, so that every GPU computes the
// same bits.  The longest chunk that still gives about one wave of pass-1 CTAs (65536 rows is 1024
// CTAs of 64 rows, 7 CTAs on each of the B200's 148 SMs), from 1024 down to 128 frames.
uint32_t iir_chunk_len(uint64_t nstreams, uint64_t nframes)
{
    uint32_t len = 1024;
    while (len > 128 && nstreams * ((nframes + len - 1) / len) < 65536)
        len /= 2;
    return len;
}



size_t iir_state_bytes(const IirView &v)
{
    return size_t(v.k.nsections) * v.nstreams * 16; // two complex64 values per section and stream
}

// A stage of the filtered iteration: the filter's view, or no sections for a stage left out.
IirView iir_stage(const sxgpu_iir *f)
{
    IirView v = {};
    if (f)
        v = f->view;
    return v;
}

} // namespace

extern "C" {

int sxgpu_iir_create(sxgpu_ctx *ctx, uint32_t nstreams, uint32_t nsections, const double *sos, sxgpu_iir **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (nstreams == 0)
        return ctx->invalid("a filter needs at least one stream");
    if (nsections < 1 || nsections > SXGPU_IIR_MAX_SECTIONS || !sos)
        return ctx->invalid("a filter has 1 to SXGPU_IIR_MAX_SECTIONS second-order sections");
    IirView v = {};
    v.nstreams = nstreams;
    v.k.nsections = nsections;
    for (uint32_t q = 0; q < nsections; q++) {
        const double *row = sos + size_t(q) * 6;
        for (int i = 0; i < 6; i++)
            if (!std::isfinite(row[i]))
                return ctx->invalid("every filter coefficient must be finite");
        if (row[3] != 1.0)
            return ctx->invalid("a0 of every section must be 1 (scipy's sos layout: b0 b1 b2 a0 a1 a2)");
        v.k.b0[q] = float(row[0]);
        v.k.b1[q] = float(row[1]);
        v.k.b2[q] = float(row[2]);
        v.k.a1[q] = float(row[4]);
        v.k.a2[q] = float(row[5]);
    }
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const std::vector<double> chain = iir_power_chain(v.k);
    std::unique_ptr<sxgpu_iir> f(new sxgpu_iir());
    f->ctx = ctx;
    cudaError_t e = dev_upload(ctx, f->state, nullptr, iir_state_bytes(v));
    if (e == cudaSuccess)
        e = dev_upload(ctx, f->powers, chain.data(), chain.size() * sizeof(double));
    v.state = f->state.get();
    f->view = v;
    return dsp_created(ctx, f, e, "cudaMalloc(filter)", out);
}

int sxgpu_iir_destroy(sxgpu_iir *f)
{
    return dsp_destroy(f);
}

int sxgpu_iir_set_state(sxgpu_iir *f, const void *h_zi, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    return state_copy(f->ctx, f->view.state, h_zi, iir_state_bytes(f->view), cudaMemcpyHostToDevice, stream);
}

int sxgpu_iir_get_state(sxgpu_iir *f, void *h_zf, sxgpu_stream stream)
{
    if (!f || !h_zf)
        return SXGPU_ERR_INVALID;
    return state_copy(f->ctx, h_zf, f->view.state, iir_state_bytes(f->view), cudaMemcpyDeviceToHost, stream);
}

int sxgpu_iir_apply(sxgpu_iir *f, void *d_cf32, uint32_t period, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = f->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("CF32 buffer must be 8-byte aligned device memory");
    if (period < 1 || period > 65536)
        return ctx->invalid("the period is 1 to 65536 frames");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const unsigned grid = unsigned((uint64_t(f->view.nstreams) + kIirStreamsPerCta - 1) / kIirStreamsPerCta);
    iir_apply_kernel<<<grid, kIirThreads, 0, call_stream(f->ctx, stream)>>>(f->view, static_cast<char *>(d_cf32), period, IirChunks{});
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

int sxgpu_iir_apply_long(sxgpu_iir *f, void *d_cf32, uint64_t nframes, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = f->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("CF32 buffer must be 8-byte aligned device memory");
    if (nframes == 0)
        return ctx->invalid("sxgpu_iir_apply_long: a block has at least one frame");
    const uint64_t nstreams = f->view.nstreams;
    if (nframes > UINT64_MAX / 8 / nstreams)
        return ctx->invalid("sxgpu_iir_apply_long: nstreams * nframes * 8 bytes overflows 64 bits");
    const uint32_t len = iir_chunk_len(nstreams, nframes);
    const uint64_t chunks = (nframes + len - 1) / len;
    const uint64_t ctas = (nstreams * chunks + kIirStreamsPerCta - 1) / kIirStreamsPerCta;
    if (ctas > uint64_t(INT32_MAX))
        return ctx->invalid("sxgpu_iir_apply_long: the block needs more CTAs than a grid holds");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(f->ctx, stream);
    char *cf32 = static_cast<char *>(d_cf32);
    if (chunks == 1) { // the whole block is chunk 0: exactly sxgpu_iir_apply
        const unsigned grid = unsigned((nstreams + kIirStreamsPerCta - 1) / kIirStreamsPerCta);
        iir_apply_kernel<<<grid, kIirThreads, 0, st>>>(f->view, cf32, uint32_t(nframes), IirChunks{});
        SX_CUDA(ctx, cudaGetLastError());
        ctx->launches++;
        return SXGPU_OK;
    }
    const uint64_t groups = (chunks + kIirGroup - 1) / kIirGroup, sequences = nstreams * groups * 2;
    const size_t edge_bytes = size_t(nstreams * chunks) * 2 * kIirDim * sizeof(float);
    const size_t total_bytes = size_t(sequences) * kIirDim * sizeof(double);
    void *scratch = nullptr;
    SX_CUDA(ctx, cudaMallocAsync(&scratch, edge_bytes + 2 * total_bytes, st));
    double *totals[2] = {reinterpret_cast<double *>(static_cast<char *>(scratch) + edge_bytes),
                         reinterpret_cast<double *>(static_cast<char *>(scratch) + edge_bytes + total_bytes)};
    IirChunks ch = {nframes, chunks, nstreams * (chunks - 1), len, static_cast<float *>(scratch)};
    IirCarry a = {f->powers.get(), ch, nullptr, totals[0], groups, sequences, 0};
    while ((1u << a.log2_len) < len)
        a.log2_len++;
    const unsigned carry_grid = unsigned((sequences * 16 + 127) / 128);
    int launches = 0;
    cudaError_t e = cudaSuccess;
    auto launched = [&]() {
        if (e == cudaSuccess)
            e = cudaGetLastError();
        launches++;
    };
    iir_apply_kernel<kIirRowsChunkEnds>
        <<<unsigned((ch.rows + kIirStreamsPerCta - 1) / kIirStreamsPerCta), kIirThreads, 0, st>>>(f->view, cf32, 0, ch);
    launched();
    iir_carry_reduce_kernel<<<carry_grid, 128, 0, st>>>(f->view, a);
    launched();
    for (uint32_t level = 0; (uint64_t(1) << level) < groups; level++) {
        a.in = a.out;
        a.out = totals[a.out == totals[0] ? 1 : 0];
        iir_carry_scan_kernel<<<carry_grid, 128, 0, st>>>(f->view, a, level);
        launched();
    }
    a.in = a.out;
    iir_carry_fixup_kernel<<<carry_grid, 128, 0, st>>>(f->view, a);
    launched();
    ch.rows = nstreams * chunks;
    iir_apply_kernel<kIirRowsChunkOut><<<unsigned(ctas), kIirThreads, 0, st>>>(f->view, cf32, 0, ch);
    launched();
    cudaFreeAsync(scratch, st);
    if (e != cudaSuccess)
        return ctx->fail(e, "sxgpu_iir_apply_long");
    ctx->launches += launches;
    return SXGPU_OK;
}

int sxgpu_bank_repeat_filtered(sxgpu_bank *bank, sxgpu_iir *pre, sxgpu_iir *post, void *d_cf32,
                               long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if ((pre && pre->ctx != ctx) || (post && post->ctx != ctx))
        return ctx->invalid("a filter belongs to another context");
    if (pre && pre == post)
        return ctx->invalid("the two stages cannot share one filter (and its state)");
    const IirView vpre = iir_stage(pre), vpost = iir_stage(post);
    if (const char *why = bank_repeat_iir_invalid(bank->st, d_cf32, vpre, vpost))
        return ctx->invalid(why);
    if (!pre && !post)
        return sxgpu_bank_repeat(bank, d_cf32, rx_time_offset_ns, stream);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const BankState &b = bank->st;
    SX_CUDA(ctx, launch_bank_iir<kBankModeRepeat>(b, static_cast<char *>(d_cf32), bank->external_capture, SX_HAS_TIME, nullptr,
                                                  rx_time_offset_ns, vpre, vpost, call_stream(bank->ctx, stream), IdentityHook()));
    ctx->launches += 2;
    ctx->frames_rx += uint64_t(b.nstreams) * b.period;
    ctx->frames_tx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

int sxgpu_bank_read_filtered(sxgpu_bank *bank, sxgpu_iir *f, void *d_cf32, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (f && f->ctx != ctx)
        return ctx->invalid("a filter belongs to another context");
    const IirView v = iir_stage(f);
    if (const char *why = bank_repeat_iir_invalid(bank->st, d_cf32, v, IirView{}))
        return ctx->invalid(why);
    if (!f)
        return sxgpu_bank_read(bank, d_cf32, stream);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const BankState &b = bank->st;
    SX_CUDA(ctx, launch_bank_iir<kBankModeRead>(b, static_cast<char *>(d_cf32), bank->external_capture, 0, nullptr, 0, v,
                                                IirView{}, call_stream(bank->ctx, stream), IdentityHook()));
    ctx->launches += 2;
    ctx->frames_rx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

int sxgpu_bank_write_filtered(sxgpu_bank *bank, sxgpu_iir *f, const void *d_cf32, int flags, const long long *d_time_ns,
                              long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = bank->ctx;
    if (f && f->ctx != ctx)
        return ctx->invalid("a filter belongs to another context");
    const IirView v = iir_stage(f);
    if (const char *why = bank_repeat_iir_invalid(bank->st, d_cf32, v, IirView{}))
        return ctx->invalid(why);
    if (!f)
        return sxgpu_bank_write(bank, d_cf32, flags, d_time_ns, rx_time_offset_ns, stream);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const BankState &b = bank->st;
    // the kernel only loads from the block in this mode
    SX_CUDA(ctx, launch_bank_iir<kBankModeWrite>(b, const_cast<char *>(static_cast<const char *>(d_cf32)), false, flags,
                                                 d_time_ns, rx_time_offset_ns, v, IirView{}, call_stream(bank->ctx, stream),
                                                 IdentityHook()));
    ctx->launches += 2;
    ctx->frames_tx += uint64_t(b.nstreams) * b.period;
    return SXGPU_OK;
}

int sxgpu_iir_device_view(sxgpu_iir *f, void *out, size_t out_bytes)
{
    if (!f || !out)
        return SXGPU_ERR_INVALID;
    if (out_bytes != sizeof(IirView))
        return f->ctx->invalid("sxgpu_iir_device_view: size mismatch (header and library disagree)");
    std::memcpy(out, &f->view, sizeof(IirView));
    return SXGPU_OK;
}

// ---- stateful FIR filters and rational resamplers (sx_fir.cuh) ------------------------------------
} // extern "C"

struct sxgpu_fir {
    sxgpu_ctx *ctx = nullptr;
    uint32_t nstreams = 0, up = 1, down = 1, g = 1, up1 = 1, down1 = 1, hp = 1, rows = 1;
    uint32_t phase = 0;       // frames fed so far mod down: the only state kept on the host
    DevPtr<float4> taps;      // [up][rows] tap tables (FirCall::taps), device memory
    DevPtr<float2> hist;      // [nstreams][hp - 1], device memory; NULL when hp == 1
};

namespace {

constexpr size_t kFirWindowBytes = 200 * 1024; // fir_apply_kernel's window stays below the 227 KB of an SM

// Outputs a call of nin frames emits from phase r: ceil((r + nin) U / D) - ceil(r U / D), or
// UINT64_MAX if that does not fit.
uint64_t fir_outputs(const sxgpu_fir *f, uint32_t r, uint64_t nin)
{
    const unsigned __int128 up = f->up, down = f->down;
    const unsigned __int128 end = ((r + (unsigned __int128)nin) * up + down - 1) / down;
    const unsigned __int128 n = end - (r * up + down - 1) / down;
    return n > UINT64_MAX ? UINT64_MAX : uint64_t(n);
}

// The geometry of a call of nin frames that emits n = fir_outputs(f, f->phase, nin) frames, without
// its buffers; `block` is the R of the data kernel (0 when n is 0) and `smem` its window in bytes.
// False when the data kernel's grid would not fit.
bool fir_call(const sxgpu_fir *f, uint64_t nin, uint64_t n, FirCall &a, int &block, size_t &smem)
{
    a.hist = f->hist.get();
    a.taps = f->taps.get();
    a.nin = nin;
    a.nout = n;
    a.c0 = (uint64_t(f->phase) * f->up + f->down - 1) / f->down;
    a.a_lo = a.c0 / f->up1;
    a.hp = f->hp;
    a.rows = f->rows;
    a.g = f->g;
    a.up1 = f->up1;
    a.down1 = f->down1;
    a.phase = f->phase;
    block = 0;
    smem = 0;
    if (n) {
        const uint64_t classes = (a.c0 + n - 1) / f->up1 - a.a_lo + 1; // class indices a the call covers
        const uint32_t e_max = (f->up1 - 1) * f->down1 / f->up1;
        for (block = classes >= 128 ? 4 : classes >= 64 ? 2 : 1;; block /= 2) {
            const uint32_t seg = uint32_t(block) * f->down1;
            a.win_len = 32 * seg + e_max + f->hp;
            a.pad = seg % 2 == 0;
            smem = (a.win_len + (a.pad ? a.win_len / seg : 0)) * sizeof(float2);
            if (smem <= kFirWindowBytes || block == 1)
                break;
        }
        a.chunks = (classes + 32 * block - 1) / (32 * block);
        if (a.chunks > uint64_t(INT32_MAX) / f->nstreams)
            return false;
    }
    return true;
}

size_t fir_hist_bytes(const sxgpu_fir *f)
{
    return size_t(f->nstreams) * (f->hp - 1) * sizeof(float2);
}

} // namespace

extern "C" {

int sxgpu_fir_create(sxgpu_ctx *ctx, uint32_t nstreams, uint32_t ntaps, const double *h, uint32_t up, uint32_t down,
                     sxgpu_fir **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (nstreams == 0 || nstreams > uint32_t(INT32_MAX))
        return ctx->invalid("a FIR filter has 1 to 2^31 - 1 streams (one CTA each for the history)");
    if (ntaps < 1 || ntaps > SXGPU_FIR_MAX_TAPS || !h)
        return ctx->invalid("a FIR filter has 1 to SXGPU_FIR_MAX_TAPS taps");
    if (up < 1 || up > SXGPU_FIR_MAX_FACTOR || down < 1 || down > SXGPU_FIR_MAX_FACTOR)
        return ctx->invalid("up and down are 1 to SXGPU_FIR_MAX_FACTOR");
    for (uint32_t i = 0; i < ntaps; i++)
        if (!std::isfinite(h[i]))
            return ctx->invalid("every FIR tap must be finite");
    std::unique_ptr<sxgpu_fir> f(new sxgpu_fir());
    f->ctx = ctx;
    f->nstreams = nstreams;
    f->up = up;
    f->down = down;
    uint32_t g = up, d = down;
    while (d) {
        const uint32_t t = g % d;
        g = d;
        d = t;
    }
    f->g = g;
    f->up1 = up / g;
    f->down1 = down / g;
    f->hp = (ntaps + up - 1) / up;
    f->rows = (kFirBlock - 1) * f->down1 + f->hp;
    // Row q of phase t's table holds, for i < kFirBlock, tap s = q - i D' of the phase in
    // accumulation order, h[t + U (hp - 1 - s)] (0 past the taps, and where that s does not exist).
    std::vector<float> taps(size_t(up) * f->rows * 4, 0.0f);
    for (uint32_t t = 0; t < up; t++)
        for (uint32_t q = 0; q < f->rows; q++)
            for (uint32_t i = 0; i < uint32_t(kFirBlock); i++) {
                if (q < i * f->down1 || q - i * f->down1 >= f->hp)
                    continue;
                const uint64_t j = t + uint64_t(up) * (f->hp - 1 - (q - i * f->down1));
                taps[(size_t(t) * f->rows + q) * 4 + i] = j < ntaps ? float(h[j]) : 0.0f;
            }
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t smem = std::min<size_t>(kFirWindowBytes, ctx->prop.sharedMemPerBlockOptin);
    for (auto kernel : {fir_apply_kernel<1>, fir_apply_kernel<2>, fir_apply_kernel<4>})
        SX_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    SX_CUDA(ctx, bank_fir_allow_smem<NoNco>(smem));
    cudaError_t e = dev_upload(ctx, f->taps, taps.data(), taps.size() * sizeof(float));
    if (e == cudaSuccess && f->hp > 1)
        e = dev_upload(ctx, f->hist, nullptr, fir_hist_bytes(f.get()));
    return dsp_created(ctx, f, e, "cudaMalloc(FIR filter)", out);
}

int sxgpu_fir_destroy(sxgpu_fir *f)
{
    return dsp_destroy(f);
}

int sxgpu_fir_output_frames(sxgpu_fir *f, uint64_t nin, uint64_t *nout)
{
    if (!f || !nout)
        return SXGPU_ERR_INVALID;
    const uint64_t n = fir_outputs(f, f->phase, nin);
    if (n == UINT64_MAX)
        return f->ctx->invalid("sxgpu_fir_output_frames: the output count overflows 64 bits");
    *nout = n;
    return SXGPU_OK;
}

int sxgpu_fir_apply(sxgpu_fir *f, const void *d_in, uint64_t nin, void *d_out, uint64_t *nout, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = f->ctx;
    if (!d_in || !d_out || reinterpret_cast<uintptr_t>(d_in) % 8 || reinterpret_cast<uintptr_t>(d_out) % 8)
        return ctx->invalid("sxgpu_fir_apply: input and output must be 8-byte aligned device memory");
    if (nin == 0)
        return ctx->invalid("sxgpu_fir_apply: a block has at least one frame");
    const uint64_t nstreams = f->nstreams;
    if (nin > UINT64_MAX / 8 / nstreams)
        return ctx->invalid("sxgpu_fir_apply: nstreams * nin * 8 bytes overflows 64 bits");
    const uint64_t n = fir_outputs(f, f->phase, nin);
    if (n > UINT64_MAX / 8 / nstreams)
        return ctx->invalid("sxgpu_fir_apply: nstreams * nout * 8 bytes overflows 64 bits");
    const uintptr_t in0 = reinterpret_cast<uintptr_t>(d_in), out0 = reinterpret_cast<uintptr_t>(d_out);
    const uint64_t in_bytes = nstreams * nin * 8, out_bytes = nstreams * n * 8;
    if (out_bytes && (in0 >= out0 ? in0 - out0 < out_bytes : out0 - in0 < in_bytes))
        return ctx->invalid("sxgpu_fir_apply: input and output overlap");

    FirCall a = {};
    int block = 0;
    size_t smem = 0;
    if (!fir_call(f, nin, n, a, block, smem))
        return ctx->invalid("sxgpu_fir_apply: the block needs more CTAs than a grid holds");
    a.in = static_cast<const float2 *>(d_in);
    a.out = static_cast<float2 *>(d_out);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(f->ctx, stream);
    int launches = 0;
    if (n) {
        const unsigned grid = unsigned(nstreams * a.chunks);
        if (block == 4)
            fir_apply_kernel<4><<<grid, 32, smem, st>>>(a);
        else if (block == 2)
            fir_apply_kernel<2><<<grid, 32, smem, st>>>(a);
        else
            fir_apply_kernel<1><<<grid, 32, smem, st>>>(a);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    if (f->hp > 1) {
        fir_history_kernel<<<unsigned(nstreams), kFirHistoryThreads, (f->hp - 1) * sizeof(float2), st>>>(a);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    ctx->launches += launches;
    f->phase = uint32_t((f->phase + nin % f->down) % f->down);
    if (nout)
        *nout = n;
    return SXGPU_OK;
}

int sxgpu_fir_get_state(sxgpu_fir *f, void *h_hist, uint32_t *phase, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = f->ctx;
    if (h_hist && f->hp > 1)
        SX_TRY(state_copy(ctx, h_hist, f->hist.get(), fir_hist_bytes(f), cudaMemcpyDeviceToHost, stream));
    if (phase)
        *phase = f->phase;
    return SXGPU_OK;
}

int sxgpu_fir_set_state(sxgpu_fir *f, const void *h_hist, uint32_t phase, sxgpu_stream stream)
{
    if (!f)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = f->ctx;
    if (phase >= f->down)
        return ctx->invalid("sxgpu_fir_set_state: the phase is below down");
    if (f->hp > 1)
        SX_TRY(state_copy(ctx, f->hist.get(), h_hist, fir_hist_bytes(f), cudaMemcpyHostToDevice, stream));
    f->phase = phase;
    return SXGPU_OK;
}

// ---- numerically controlled oscillators (sx_nco.cuh) ---------------------------------------------
} // extern "C"

struct sxgpu_nco {
    sxgpu_ctx *ctx = nullptr;
    uint32_t nstreams = 0;
    DevPtr<char> mem; // one allocation: the tables, then the phases, then the increments
    NcoView view = {};
};

namespace {

// inc = rint(f 2^32) mod 2^32 for every stream (f NULL: all 0), or why a frequency is refused.
const char *nco_increments(uint32_t nstreams, const double *freq, std::vector<uint32_t> &inc)
{
    inc.assign(nstreams, 0);
    for (uint32_t s = 0; freq && s < nstreams; s++) {
        if (!std::isfinite(freq[s]) || std::fabs(freq[s]) > 0.5)
            return "an oscillator's frequency is finite and within -0.5 .. 0.5 cycles per sample";
        inc[s] = uint32_t(uint64_t(std::llrint(freq[s] * 4294967296.0)));
    }
    return nullptr;
}

// A[k] = e^{j 2 pi k / 1024}, then B[k] = e^{j 2 pi k / 2^20}: libm's double cos and sin, rounded
// once.  The channelizers' twiddles are A conjugated.
std::vector<float2> nco_tables()
{
    std::vector<float2> tab(2 * kNcoTableSize);
    for (int k = 0; k < kNcoTableSize; k++) {
        const double a = 2.0 * M_PI * k / 1024.0, b = 2.0 * M_PI * k / 1048576.0;
        tab[k] = make_float2(float(std::cos(a)), float(std::sin(a)));
        tab[kNcoTableSize + k] = make_float2(float(std::cos(b)), float(std::sin(b)));
    }
    return tab;
}

} // namespace

extern "C" {

int sxgpu_nco_create(sxgpu_ctx *ctx, uint32_t nstreams, const double *freq, sxgpu_nco **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (nstreams == 0 || nstreams > uint32_t(INT32_MAX))
        return ctx->invalid("an oscillator has 1 to 2^31 - 1 streams");
    std::vector<uint32_t> inc;
    if (const char *why = nco_increments(nstreams, freq, inc))
        return ctx->invalid(why);
    const std::vector<float2> tab = nco_tables();
    const size_t tab_bytes = tab.size() * sizeof(float2), state_bytes = size_t(nstreams) * sizeof(uint32_t);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, bank_fir_allow_smem<NcoView>(std::min<size_t>(kFirWindowBytes, ctx->prop.sharedMemPerBlockOptin)));
    std::unique_ptr<sxgpu_nco> n(new sxgpu_nco());
    n->ctx = ctx;
    n->nstreams = nstreams;
    std::vector<char> img(tab_bytes + 2 * state_bytes, 0); // the phases start at 0
    std::memcpy(img.data(), tab.data(), tab_bytes);
    std::memcpy(img.data() + tab_bytes + state_bytes, inc.data(), state_bytes);
    const cudaError_t e = dev_upload(ctx, n->mem, img.data(), img.size());
    char *mem = n->mem.get();
    n->view = NcoView{reinterpret_cast<const float2 *>(mem), reinterpret_cast<uint32_t *>(mem + tab_bytes),
                      reinterpret_cast<uint32_t *>(mem + tab_bytes + state_bytes)};
    return dsp_created(ctx, n, e, "cudaMalloc(oscillator)", out);
}

int sxgpu_nco_destroy(sxgpu_nco *n)
{
    return dsp_destroy(n);
}

int sxgpu_nco_apply(sxgpu_nco *n, void *d_cf32, uint64_t nframes, sxgpu_stream stream)
{
    if (!n)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = n->ctx;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 8)
        return ctx->invalid("sxgpu_nco_apply: the block must be 8-byte aligned device memory");
    if (nframes == 0)
        return ctx->invalid("sxgpu_nco_apply: a block has at least one frame");
    if (nframes > UINT64_MAX / 8 / n->nstreams)
        return ctx->invalid("sxgpu_nco_apply: nstreams * nframes * 8 bytes overflows 64 bits");
    const uint64_t total = uint64_t(n->nstreams) * nframes, ctas = (total + kNcoTile - 1) / kNcoTile;
    if (ctas > uint64_t(INT32_MAX))
        return ctx->invalid("sxgpu_nco_apply: the block needs more CTAs than a grid holds");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(n->ctx, stream);
    nco_apply_kernel<<<unsigned(ctas), kNcoThreads, 0, st>>>(n->view, static_cast<float2 *>(d_cf32), nframes, total,
                                                             1.0 / double(nframes));
    SX_CUDA(ctx, cudaGetLastError());
    nco_advance_kernel<<<per_stream_grid(n->nstreams, 256), 256, 0, st>>>(n->view, n->nstreams, uint32_t(nframes));
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches += 2;
    return SXGPU_OK;
}

int sxgpu_nco_set_frequencies(sxgpu_nco *n, const double *h_freq, sxgpu_stream stream)
{
    if (!n)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = n->ctx;
    std::vector<uint32_t> inc;
    if (const char *why = nco_increments(n->nstreams, h_freq, inc))
        return ctx->invalid(why);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(n->ctx, stream);
    SX_CUDA(ctx, cudaMemcpyAsync(n->view.inc, inc.data(), inc.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int sxgpu_nco_get_state(sxgpu_nco *n, uint32_t *h_phase, uint32_t *h_inc, sxgpu_stream stream)
{
    if (!n)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = n->ctx;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(n->ctx, stream);
    const size_t bytes = size_t(n->nstreams) * sizeof(uint32_t);
    if (h_phase)
        SX_CUDA(ctx, cudaMemcpyAsync(h_phase, n->view.phase, bytes, cudaMemcpyDeviceToHost, st));
    if (h_inc)
        SX_CUDA(ctx, cudaMemcpyAsync(h_inc, n->view.inc, bytes, cudaMemcpyDeviceToHost, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

int sxgpu_nco_set_state(sxgpu_nco *n, const uint32_t *h_phase, const uint32_t *h_inc, sxgpu_stream stream)
{
    if (!n)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = n->ctx;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(n->ctx, stream);
    const size_t bytes = size_t(n->nstreams) * sizeof(uint32_t);
    if (h_phase)
        SX_CUDA(ctx, cudaMemcpyAsync(n->view.phase, h_phase, bytes, cudaMemcpyHostToDevice, st));
    if (h_inc)
        SX_CUDA(ctx, cudaMemcpyAsync(n->view.inc, h_inc, bytes, cudaMemcpyHostToDevice, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    return SXGPU_OK;
}

// ---- the stream bank's FIR halves, with or without an oscillator (sx_bank.cuh) -------------------
} // extern "C"

namespace {

// Why a FIR half's filter is refused (nullptr: it is not).
const char *bank_fir_invalid(const sxgpu_bank *bank, const sxgpu_fir *f)
{
    if (!f || f->ctx != bank->ctx)
        return "the FIR filter is NULL or belongs to another context";
    if (f->nstreams != bank->st.nstreams)
        return "a filter must have as many streams as the bank";
    return nullptr;
}

// Why a half's oscillator is refused (nullptr: it is not).
const char *bank_nco_invalid(const sxgpu_bank *bank, const sxgpu_nco *n)
{
    if (!n || n->ctx != bank->ctx)
        return "the oscillator is NULL or belongs to another context";
    if (n->nstreams != bank->st.nstreams)
        return "an oscillator must have as many streams as the bank";
    return nullptr;
}

// sxgpu_bank_read_fir (nco: NoNco) and sxgpu_bank_read_ddc (nco: the oscillator's NcoView), after
// the entry point `name` has checked the filter and the oscillator.
template <class Nco>
int bank_read_fir(sxgpu_bank *bank, sxgpu_fir *f, const Nco &nco, void *d_out, uint64_t *nout, sxgpu_stream stream,
                  const char *name)
{
    sxgpu_ctx *ctx = bank->ctx;
    auto refuse = [&](const char *why) { return ctx->invalid((std::string(name) + ": " + why).c_str()); };
    if (!d_out || reinterpret_cast<uintptr_t>(d_out) % 8)
        return refuse("the output must be 8-byte aligned device memory");
    const BankState &b = bank->st;
    const uint64_t n = fir_outputs(f, f->phase, b.period);
    if (n > UINT64_MAX / 8 / b.nstreams)
        return refuse("nstreams * nout * 8 bytes overflows 64 bits");
    FirCall a = {};
    int block = 0;
    size_t smem = 0;
    if (!fir_call(f, b.period, n, a, block, smem))
        return refuse("the period needs more CTAs than a grid holds");
    a.out = static_cast<float2 *>(d_out);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    const bool ext = bank->external_capture;
    SX_CUDA(ctx, launch_bank_plan<kBankModeRead>(b, nullptr, 0, nullptr, 0, st));
    int launches = 1;
    if (n) {
        SX_CUDA(ctx, launch_bank_fir<kBankModeRead>(b, a, block, smem, ext, nco, st));
        launches++;
    }
    if (f->hp > 1 || !ext || !std::is_same<Nco, NoNco>::value) { // with an oscillator the tail advances the phases
        bank_fir_read_tail_kernel<<<b.nstreams, kFirHistoryThreads, (f->hp - 1) * sizeof(float2), st>>>(b, a, ext, nco);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    ctx->launches += launches;
    ctx->frames_rx += uint64_t(b.nstreams) * b.period;
    f->phase = uint32_t((f->phase + b.period % f->down) % f->down);
    if (nout)
        *nout = n;
    return SXGPU_OK;
}

// sxgpu_bank_write_fir (nco: NoNco) and sxgpu_bank_write_duc (nco: the oscillator's NcoView), after
// the entry point `name` has checked the filter and the oscillator.
template <class Nco>
int bank_write_fir(sxgpu_bank *bank, sxgpu_fir *f, const Nco &nco, const void *d_in, uint64_t nin, int flags,
                   const long long *d_time_ns, long long rx_time_offset_ns, sxgpu_stream stream, const char *name)
{
    sxgpu_ctx *ctx = bank->ctx;
    auto refuse = [&](const char *why) { return ctx->invalid((std::string(name) + ": " + why).c_str()); };
    if (!d_in || reinterpret_cast<uintptr_t>(d_in) % 8)
        return refuse("the input must be 8-byte aligned device memory");
    const BankState &b = bank->st;
    if (nin > UINT64_MAX / 8 / b.nstreams)
        return refuse("nstreams * nin * 8 bytes overflows 64 bits");
    if (fir_outputs(f, f->phase, nin) != b.period)
        return refuse("the filter must emit exactly one period from nin frames");
    FirCall a = {};
    int block = 0;
    size_t smem = 0;
    if (!fir_call(f, nin, b.period, a, block, smem))
        return refuse("the block needs more CTAs than a grid holds");
    a.in = static_cast<const float2 *>(d_in);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    SX_CUDA(ctx, launch_bank_plan<kBankModeWrite>(b, nullptr, flags, d_time_ns, rx_time_offset_ns, st));
    SX_CUDA(ctx, launch_bank_fir<kBankModeWrite>(b, a, block, smem, false, nco, st));
    int launches = 2;
    if (f->hp > 1 || !std::is_same<Nco, NoNco>::value) { // with an oscillator the tail advances the phases
        fir_history_kernel<<<b.nstreams, kFirHistoryThreads, (f->hp - 1) * sizeof(float2), st>>>(a, nco, b.period);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    ctx->launches += launches;
    ctx->frames_tx += uint64_t(b.nstreams) * b.period;
    f->phase = uint32_t((f->phase + nin % f->down) % f->down);
    return SXGPU_OK;
}

} // namespace

extern "C" {

int sxgpu_bank_read_fir(sxgpu_bank *bank, sxgpu_fir *f, void *d_out, uint64_t *nout, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    if (const char *why = bank_fir_invalid(bank, f))
        return bank->ctx->invalid(why);
    return bank_read_fir(bank, f, NoNco{}, d_out, nout, stream, "sxgpu_bank_read_fir");
}

int sxgpu_bank_read_ddc(sxgpu_bank *bank, sxgpu_nco *nco, sxgpu_fir *f, void *d_out, uint64_t *nout, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    if (const char *why = bank_nco_invalid(bank, nco))
        return bank->ctx->invalid(why);
    if (const char *why = bank_fir_invalid(bank, f))
        return bank->ctx->invalid(why);
    return bank_read_fir(bank, f, nco->view, d_out, nout, stream, "sxgpu_bank_read_ddc");
}

int sxgpu_bank_write_fir(sxgpu_bank *bank, sxgpu_fir *f, const void *d_in, uint64_t nin, int flags,
                         const long long *d_time_ns, long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    if (const char *why = bank_fir_invalid(bank, f))
        return bank->ctx->invalid(why);
    return bank_write_fir(bank, f, NoNco{}, d_in, nin, flags, d_time_ns, rx_time_offset_ns, stream, "sxgpu_bank_write_fir");
}

int sxgpu_bank_write_duc(sxgpu_bank *bank, sxgpu_fir *f, sxgpu_nco *nco, const void *d_in, uint64_t nin, int flags,
                         const long long *d_time_ns, long long rx_time_offset_ns, sxgpu_stream stream)
{
    if (!bank)
        return SXGPU_ERR_INVALID;
    if (const char *why = bank_fir_invalid(bank, f))
        return bank->ctx->invalid(why);
    if (const char *why = bank_nco_invalid(bank, nco))
        return bank->ctx->invalid(why);
    return bank_write_fir(bank, f, nco->view, d_in, nin, flags, d_time_ns, rx_time_offset_ns, stream, "sxgpu_bank_write_duc");
}

// ---- polyphase DFT channelizers (sx_chan.cuh) -------------------------------------------------
} // extern "C"

struct sxgpu_chan {
    sxgpu_ctx *ctx = nullptr;
    uint32_t nstreams = 0, m = 2, log2m = 1, down = 1, ntaps = 1;
    uint32_t phase = 0;     // frames fed so far mod M: the only state kept on the host
    DevPtr<float2> mem;     // one allocation: the twiddles [1024], then the taps [ntaps]
    DevPtr<float2> hist;    // [nstreams][ntaps - 1], device memory; NULL when ntaps == 1
};

namespace {

constexpr size_t kChanSmemBytes = 200 * 1024; // chan_apply_kernel's shared memory, below the 227 KB of an SM
constexpr uint32_t kChanTargetThreads = 512;

// ceil((r + nin) / D) - ceil(r / D): with D dividing M, what a stream whose frame count is r mod M emits.
uint64_t chan_outputs(const sxgpu_chan *c, uint32_t r, uint64_t nin)
{
    const unsigned __int128 d = c->down;
    return uint64_t((r + (unsigned __int128)nin + d - 1) / d - (r + d - 1) / d);
}

// The geometry of a call of nin frames emitting n = chan_outputs(c, c->phase, nin) frames, without
// its buffers, and the kernel's threads and shared memory.  False when the grid would not fit.
bool chan_call(const sxgpu_chan *c, uint64_t nin, uint64_t n, ChanCall &a, uint32_t &threads, size_t &smem)
{
    const uint32_t M = c->m, D = c->down;
    a.hist = c->hist.get();
    a.tw = c->mem.get();
    a.taps = reinterpret_cast<const float *>(c->mem.get() + kNcoTableSize);
    a.nin = nin;
    a.nout = n;
    a.m = M;
    a.log2m = c->log2m;
    a.down = D;
    a.ntaps = c->ntaps;
    a.e0 = (D - c->phase % D) % D;
    a.rot0 = (c->phase + a.e0) % M;
    threads = 0;
    smem = 0;
    if (n == 0)
        return true;
    // As many groups as fill the target thread count (a whole branch set when M is above it),
    // fewer when the call has fewer outputs or the window would not fit.
    uint32_t g = std::max<uint32_t>(1, kChanTargetThreads / M);
    while (g > 1 && uint64_t(kChanBlock) * (g / 2) >= n)
        g /= 2;
    for (;; g /= 2) {
        const uint32_t t = kChanBlock * g;
        a.win_len = (t - 1) * D + c->ntaps;
        smem = size_t(std::max<uint64_t>(a.win_len, uint64_t(t) * (M + 1))) * sizeof(float2);
        if (smem <= kChanSmemBytes || g == 1)
            break;
    }
    a.groups = g;
    threads = M * g;
    const uint64_t t = kChanBlock * g;
    a.tiles = (n + t - 1) / t;
    return a.tiles <= uint64_t(INT32_MAX) / c->nstreams;
}

size_t chan_hist_bytes(const sxgpu_chan *c)
{
    return size_t(c->nstreams) * (c->ntaps - 1) * sizeof(float2);
}

} // namespace

extern "C" {

int sxgpu_chan_create(sxgpu_ctx *ctx, uint32_t nstreams, uint32_t channels, uint32_t down, uint32_t ntaps,
                      const double *h, sxgpu_chan **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (channels < 2 || channels > SXGPU_CHAN_MAX_CHANNELS || (channels & (channels - 1)))
        return ctx->invalid("a channelizer has a power of two of 2 to SXGPU_CHAN_MAX_CHANNELS channels");
    if (nstreams == 0 || uint64_t(nstreams) * channels > uint64_t(INT32_MAX))
        return ctx->invalid("a channelizer has 1 to (2^31 - 1) / channels streams");
    if (down == 0 || channels % down)
        return ctx->invalid("a channelizer's decimation divides its channel count");
    if (ntaps < 1 || ntaps > SXGPU_CHAN_MAX_TAPS || ntaps > 32 * channels || !h)
        return ctx->invalid("a channelizer has 1 to min(SXGPU_CHAN_MAX_TAPS, 32 channels) taps");
    for (uint32_t i = 0; i < ntaps; i++)
        if (!std::isfinite(h[i]))
            return ctx->invalid("every channelizer tap must be finite");
    std::unique_ptr<sxgpu_chan> c(new sxgpu_chan());
    c->ctx = ctx;
    c->nstreams = nstreams;
    c->m = channels;
    while ((1u << c->log2m) < channels)
        c->log2m++;
    c->down = down;
    c->ntaps = ntaps;
    // The twiddles: the oscillator's coarse table conjugated, then the taps rounded once.
    std::vector<float2> tw = nco_tables();
    tw.resize(kNcoTableSize);
    for (float2 &w : tw)
        w.y = -w.y;
    std::vector<float> taps(ntaps);
    for (uint32_t i = 0; i < ntaps; i++)
        taps[i] = float(h[i]);
    const size_t tw_bytes = tw.size() * sizeof(float2), taps_bytes = taps.size() * sizeof(float);
    std::vector<char> img(tw_bytes + taps_bytes);
    std::memcpy(img.data(), tw.data(), tw_bytes);
    std::memcpy(img.data() + tw_bytes, taps.data(), taps_bytes);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaFuncSetAttribute(chan_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int(std::min<size_t>(kChanSmemBytes, ctx->prop.sharedMemPerBlockOptin))));
    SX_CUDA(ctx, cudaFuncSetAttribute(fir_history_kernel<NoNco>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int((kChanMaxTaps - 1) * sizeof(float2))));
    cudaError_t e = dev_upload(ctx, c->mem, img.data(), img.size());
    if (e == cudaSuccess && ntaps > 1)
        e = dev_upload(ctx, c->hist, nullptr, chan_hist_bytes(c.get()));
    return dsp_created(ctx, c, e, "cudaMalloc(channelizer)", out);
}

int sxgpu_chan_destroy(sxgpu_chan *c)
{
    return dsp_destroy(c);
}

int sxgpu_chan_output_frames(sxgpu_chan *c, uint64_t nin, uint64_t *nout)
{
    if (!c || !nout)
        return SXGPU_ERR_INVALID;
    *nout = chan_outputs(c, c->phase, nin);
    return SXGPU_OK;
}

int sxgpu_chan_apply(sxgpu_chan *c, const void *d_in, uint64_t nin, void *d_out, uint64_t *nout, sxgpu_stream stream)
{
    if (!c)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = c->ctx;
    if (!d_in || !d_out || reinterpret_cast<uintptr_t>(d_in) % 8 || reinterpret_cast<uintptr_t>(d_out) % 8)
        return ctx->invalid("sxgpu_chan_apply: input and output must be 8-byte aligned device memory");
    if (nin == 0)
        return ctx->invalid("sxgpu_chan_apply: a block has at least one frame");
    const uint64_t nstreams = c->nstreams, rows = nstreams * c->m;
    if (nin > UINT64_MAX / 8 / nstreams)
        return ctx->invalid("sxgpu_chan_apply: nstreams * nin * 8 bytes overflows 64 bits");
    const uint64_t n = chan_outputs(c, c->phase, nin);
    if (n > UINT64_MAX / 8 / rows)
        return ctx->invalid("sxgpu_chan_apply: nstreams * channels * nout * 8 bytes overflows 64 bits");
    const uintptr_t in0 = reinterpret_cast<uintptr_t>(d_in), out0 = reinterpret_cast<uintptr_t>(d_out);
    const uint64_t in_bytes = nstreams * nin * 8, out_bytes = rows * n * 8;
    if (out_bytes && (in0 >= out0 ? in0 - out0 < out_bytes : out0 - in0 < in_bytes))
        return ctx->invalid("sxgpu_chan_apply: input and output overlap");

    ChanCall a = {};
    uint32_t threads = 0;
    size_t smem = 0;
    if (!chan_call(c, nin, n, a, threads, smem))
        return ctx->invalid("sxgpu_chan_apply: the block needs more CTAs than a grid holds");
    a.in = static_cast<const float2 *>(d_in);
    a.out = static_cast<float2 *>(d_out);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(c->ctx, stream);
    int launches = 0;
    if (n) {
        chan_apply_kernel<<<unsigned(nstreams * a.tiles), threads, smem, st>>>(a);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    if (c->ntaps > 1) {
        // fir_history_kernel keeps the last hp - 1 frames of buf = hist ++ in: the same history.
        FirCall hc = {};
        hc.in = a.in;
        hc.hist = c->hist.get();
        hc.nin = nin;
        hc.hp = c->ntaps;
        fir_history_kernel<<<unsigned(nstreams), kFirHistoryThreads, (c->ntaps - 1) * sizeof(float2), st>>>(hc);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    ctx->launches += launches;
    c->phase = uint32_t((c->phase + nin % c->m) % c->m);
    if (nout)
        *nout = n;
    return SXGPU_OK;
}

int sxgpu_chan_get_state(sxgpu_chan *c, void *h_hist, uint32_t *phase, sxgpu_stream stream)
{
    if (!c)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = c->ctx;
    if (h_hist && c->ntaps > 1)
        SX_TRY(state_copy(ctx, h_hist, c->hist.get(), chan_hist_bytes(c), cudaMemcpyDeviceToHost, stream));
    if (phase)
        *phase = c->phase;
    return SXGPU_OK;
}

int sxgpu_chan_set_state(sxgpu_chan *c, const void *h_hist, uint32_t phase, sxgpu_stream stream)
{
    if (!c)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = c->ctx;
    if (phase >= c->m)
        return ctx->invalid("sxgpu_chan_set_state: the phase is below the channel count");
    if (c->ntaps > 1)
        SX_TRY(state_copy(ctx, c->hist.get(), h_hist, chan_hist_bytes(c), cudaMemcpyHostToDevice, stream));
    c->phase = phase;
    return SXGPU_OK;
}

// ---- polyphase synthesis channelizers (sx_chan.cuh) -------------------------------------------
} // extern "C"

struct sxgpu_chan_synth {
    sxgpu_ctx *ctx = nullptr;
    uint32_t nstreams = 0, m = 2, log2m = 1, up = 1, log2up = 0, ntaps = 1, hp = 1;
    uint32_t phase = 0;     // input frames fed so far mod M / D: the only state kept on the host
    DevPtr<float2> mem;     // one allocation: the twiddles [1024], then the taps [ntaps]
    DevPtr<float2> hist;    // [nstreams][M][hp - 1], device memory; NULL when hp == 1
};

namespace {

constexpr size_t kChanSynthSmemBytes = 96 * 1024; // two CTAs of chan_synth_kernel fit an SM's 227 KB
constexpr uint32_t kChanSynthMaxThreads = 1024;

// The geometry of a call of nin frames per channel, without its buffers, and the kernel's threads
// and shared memory.  False when the grid would not fit.
bool chan_synth_call(const sxgpu_chan_synth *c, uint64_t nin, ChanSynthCall &a, uint32_t &threads, size_t &smem)
{
    const uint32_t M = c->m, D = c->up;
    a.hist = c->hist.get();
    a.tw = c->mem.get();
    a.taps = reinterpret_cast<const float *>(c->mem.get() + kNcoTableSize);
    a.nin = nin;
    a.m = M;
    a.log2m = c->log2m;
    a.log2up = c->log2up;
    a.ntaps = c->ntaps;
    a.hp = c->hp;
    a.rot0 = (c->phase * D) % M;
    // As many input frames per tile as the threads can keep the outputs of (fewer for a short call),
    // so that the hp - 1 frames each tile transforms again are few against its own.
    uint32_t b = kChanSynthBlock * kChanSynthMaxThreads / D;
    while (b > 1 && b / 2 >= nin)
        b /= 2;
    a.frames = b;
    threads = std::max<uint32_t>(32, b * D / kChanSynthBlock);
    const size_t row = size_t(M + 1) * sizeof(float2);
    a.chunk = uint32_t(std::max<size_t>(1, std::min<size_t>(b + c->hp - 1, kChanSynthSmemBytes / row)));
    smem = a.chunk * row;
    a.tiles = (nin + b - 1) / b;
    return a.tiles <= uint64_t(INT32_MAX) / c->nstreams;
}

size_t chan_synth_hist_bytes(const sxgpu_chan_synth *c)
{
    return size_t(c->nstreams) * c->m * (c->hp - 1) * sizeof(float2);
}

} // namespace

extern "C" {

int sxgpu_chan_synth_create(sxgpu_ctx *ctx, uint32_t nstreams, uint32_t channels, uint32_t up, uint32_t ntaps,
                            const double *h, sxgpu_chan_synth **out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (channels < 2 || channels > SXGPU_CHAN_MAX_CHANNELS || (channels & (channels - 1)))
        return ctx->invalid("a synthesizer has a power of two of 2 to SXGPU_CHAN_MAX_CHANNELS channels");
    if (nstreams == 0 || uint64_t(nstreams) * channels > uint64_t(INT32_MAX))
        return ctx->invalid("a synthesizer has 1 to (2^31 - 1) / channels streams");
    if (up == 0 || channels % up)
        return ctx->invalid("a synthesizer's interpolation divides its channel count");
    if (ntaps < 1 || ntaps > SXGPU_CHAN_MAX_TAPS || ntaps > 32 * channels || !h)
        return ctx->invalid("a synthesizer has 1 to min(SXGPU_CHAN_MAX_TAPS, 32 channels) taps");
    for (uint32_t i = 0; i < ntaps; i++)
        if (!std::isfinite(h[i]))
            return ctx->invalid("every synthesizer tap must be finite");
    std::unique_ptr<sxgpu_chan_synth> c(new sxgpu_chan_synth());
    c->ctx = ctx;
    c->nstreams = nstreams;
    c->m = channels;
    while ((1u << c->log2m) < channels)
        c->log2m++;
    c->up = up;
    while ((1u << c->log2up) < up)
        c->log2up++;
    c->ntaps = ntaps;
    c->hp = (ntaps + up - 1) / up;
    // The twiddles: the oscillator's coarse table as it is, then the taps rounded once.
    std::vector<float2> tw = nco_tables();
    tw.resize(kNcoTableSize);
    std::vector<float> taps(ntaps);
    for (uint32_t i = 0; i < ntaps; i++)
        taps[i] = float(h[i]);
    const size_t tw_bytes = tw.size() * sizeof(float2), taps_bytes = taps.size() * sizeof(float);
    std::vector<char> img(tw_bytes + taps_bytes);
    std::memcpy(img.data(), tw.data(), tw_bytes);
    std::memcpy(img.data() + tw_bytes, taps.data(), taps_bytes);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaFuncSetAttribute(chan_synth_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int(std::min<size_t>(kChanSynthSmemBytes, ctx->prop.sharedMemPerBlockOptin))));
    SX_CUDA(ctx, cudaFuncSetAttribute(fir_history_kernel<NoNco>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      int((kChanMaxTaps - 1) * sizeof(float2))));
    cudaError_t e = dev_upload(ctx, c->mem, img.data(), img.size());
    if (e == cudaSuccess && c->hp > 1)
        e = dev_upload(ctx, c->hist, nullptr, chan_synth_hist_bytes(c.get()));
    return dsp_created(ctx, c, e, "cudaMalloc(synthesizer)", out);
}

int sxgpu_chan_synth_destroy(sxgpu_chan_synth *s)
{
    return dsp_destroy(s);
}

int sxgpu_chan_synth_apply(sxgpu_chan_synth *s, const void *d_in, uint64_t nin, void *d_out, sxgpu_stream stream)
{
    if (!s)
        return SXGPU_ERR_INVALID;
    sxgpu_ctx *ctx = s->ctx;
    if (!d_in || !d_out || reinterpret_cast<uintptr_t>(d_in) % 8 || reinterpret_cast<uintptr_t>(d_out) % 8)
        return ctx->invalid("sxgpu_chan_synth_apply: input and output must be 8-byte aligned device memory");
    if (nin == 0)
        return ctx->invalid("sxgpu_chan_synth_apply: a block has at least one frame");
    const uint64_t nstreams = s->nstreams, rows = nstreams * s->m;
    if (nin > UINT64_MAX / 8 / rows)
        return ctx->invalid("sxgpu_chan_synth_apply: nstreams * channels * nin * 8 bytes overflows 64 bits");
    if (nin > UINT64_MAX / 8 / nstreams / s->up)
        return ctx->invalid("sxgpu_chan_synth_apply: nstreams * nin * up * 8 bytes overflows 64 bits");
    const uintptr_t in0 = reinterpret_cast<uintptr_t>(d_in), out0 = reinterpret_cast<uintptr_t>(d_out);
    const uint64_t in_bytes = rows * nin * 8, out_bytes = nstreams * nin * s->up * 8;
    if (in0 >= out0 ? in0 - out0 < out_bytes : out0 - in0 < in_bytes)
        return ctx->invalid("sxgpu_chan_synth_apply: input and output overlap");

    ChanSynthCall a = {};
    uint32_t threads = 0;
    size_t smem = 0;
    if (!chan_synth_call(s, nin, a, threads, smem))
        return ctx->invalid("sxgpu_chan_synth_apply: the block needs more CTAs than a grid holds");
    a.in = static_cast<const float2 *>(d_in);
    a.out = static_cast<float2 *>(d_out);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    chan_synth_kernel<<<unsigned(nstreams * a.tiles), threads, smem, st>>>(a);
    SX_CUDA(ctx, cudaGetLastError());
    int launches = 1;
    if (s->hp > 1) {
        // Each of the nstreams * M channel rows keeps its last hp - 1 raw inputs, as a FIR filter's.
        FirCall hc = {};
        hc.in = a.in;
        hc.hist = s->hist.get();
        hc.nin = nin;
        hc.hp = s->hp;
        fir_history_kernel<<<unsigned(rows), kFirHistoryThreads, (s->hp - 1) * sizeof(float2), st>>>(hc);
        SX_CUDA(ctx, cudaGetLastError());
        launches++;
    }
    ctx->launches += launches;
    const uint32_t period = s->m / s->up;
    s->phase = uint32_t((s->phase + nin % period) % period);
    return SXGPU_OK;
}

int sxgpu_chan_synth_get_state(sxgpu_chan_synth *s, void *h_hist, uint32_t *phase, sxgpu_stream stream)
{
    if (!s)
        return SXGPU_ERR_INVALID;
    if (h_hist && s->hp > 1)
        SX_TRY(state_copy(s->ctx, h_hist, s->hist.get(), chan_synth_hist_bytes(s), cudaMemcpyDeviceToHost, stream));
    if (phase)
        *phase = s->phase;
    return SXGPU_OK;
}

int sxgpu_chan_synth_set_state(sxgpu_chan_synth *s, const void *h_hist, uint32_t phase, sxgpu_stream stream)
{
    if (!s)
        return SXGPU_ERR_INVALID;
    if (phase >= s->m / s->up)
        return s->ctx->invalid("sxgpu_chan_synth_set_state: the phase is below channels / up");
    if (s->hp > 1)
        SX_TRY(state_copy(s->ctx, s->hist.get(), h_hist, chan_synth_hist_bytes(s), cudaMemcpyHostToDevice, stream));
    s->phase = phase;
    return SXGPU_OK;
}

int sxgpu_fill_silence(sxgpu_ctx *ctx, void *d_i2s, size_t offset, size_t length,
                       sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (length == 0)
        return SXGPU_OK;
    if (!d_i2s || reinterpret_cast<uintptr_t>(d_i2s) % 8)
        return ctx->invalid("I2S buffer must be 8-byte aligned");
    if (frames_overflow(offset, length))
        return ctx->invalid("offset + length overflows");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    int block = 256;
    uint64_t ctas = (length + block - 1) / block;
    int grid = int(std::min<uint64_t>(ctas, uint64_t(ctx->prop.multiProcessorCount) * 8));
    fill_silence_kernel<<<grid, block, 0, st>>>(static_cast<char *>(d_i2s) + offset * 8, length);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

int sxgpu_convert_rx_buffer_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                 void *h_dest, size_t dest_offset, size_t length)
{
    int r = convert_host<RxCf32>(ctx, h_src, src_offset, h_dest, dest_offset, length, 0.0f,
                                 ctx ? ctx->rx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_rx_buffer_host_gated(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                       size_t dest_offset, size_t length, const volatile uint64_t *frames_ready,
                                       size_t *converted)
{
    if (!frames_ready)
        return ctx ? ctx->invalid("gated conversion needs a progress counter") : SXGPU_ERR_INVALID;
    size_t done = 0;
    int r = convert_host<RxCf32>(ctx, h_src, src_offset, h_dest, dest_offset, length, 0.0f, ctx ? ctx->rx_variant : 0,
                                 frames_ready, &done);
    if (converted)
        *converted = done;
    if (r == SXGPU_OK)
        ctx->frames_rx += done;
    return r;
}

int sxgpu_convert_tx_buffer_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                 void *h_dest, size_t dest_offset, size_t length,
                                 float tx_threshold2)
{
    int r = convert_host<TxCf32>(ctx, h_src, src_offset, h_dest, dest_offset, length,
                                 tx_threshold2, ctx ? ctx->tx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_convert_rx_buffer_cs16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                      void *h_dest, size_t dest_offset, size_t length)
{
    int r = convert_host<RxCs16>(ctx, h_src, src_offset, h_dest, dest_offset, length, 0.0f,
                                 ctx ? ctx->rx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_tx_buffer_cs16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                      void *h_dest, size_t dest_offset, size_t length,
                                      float tx_threshold2)
{
    int r = convert_host<TxCs16>(ctx, h_src, src_offset, h_dest, dest_offset, length,
                                 tx_threshold2, ctx ? ctx->tx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_convert_rx_buffer_s16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                     size_t dest_offset, size_t length)
{
    int r = convert_host<RxS16Cf32>(ctx, h_src, src_offset, h_dest, dest_offset, length, 0.0f,
                                    ctx ? ctx->rx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_rx += length;
    return r;
}

int sxgpu_convert_tx_buffer_s16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                     size_t dest_offset, size_t length, float tx_threshold2)
{
    int r = convert_host<TxCf32S16>(ctx, h_src, src_offset, h_dest, dest_offset, length, tx_threshold2,
                                    ctx ? ctx->tx_variant : 0);
    if (r == SXGPU_OK)
        ctx->frames_tx += length;
    return r;
}

int sxgpu_stats_words(sxgpu_ctx *ctx, const void *d_words, size_t nwords, uint64_t base_index,
                      sxgpu_stats *h_out, sxgpu_stream stream)
{
    if (!ctx || !h_out)
        return SXGPU_ERR_INVALID;
    std::memset(h_out, 0, sizeof *h_out);
    if (nwords == 0)
        return SXGPU_OK;
    if (!d_words || reinterpret_cast<uintptr_t>(d_words) % 4)
        return ctx->invalid("word buffer must be 4-byte aligned");
    std::lock_guard<std::mutex> lock(ctx->stats_mutex);
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    SX_CUDA(ctx, cudaMemsetAsync(ctx->d_stats, 0, sizeof(StatsAcc), st));
    int block = 256;
    uint64_t ctas = (nwords + block - 1) / block;
    int grid = int(std::min<uint64_t>(ctas, uint64_t(ctx->prop.multiProcessorCount) * 8));
    stats_kernel<<<grid, block, 0, st>>>(static_cast<const uint32_t *>(d_words), nwords,
                                        base_index, ctx->d_stats);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    SX_CUDA(ctx, cudaMemcpyAsync(ctx->h_stats, ctx->d_stats, sizeof(StatsAcc),
                                 cudaMemcpyDeviceToHost, st));
    SX_CUDA(ctx, cudaStreamSynchronize(st));
    h_out->sum = ctx->h_stats->sum;
    h_out->wsum = ctx->h_stats->wsum;
    h_out->x = ctx->h_stats->x;
    h_out->count = nwords;
    h_out->tx_on = ctx->h_stats->tx_on;
    h_out->rail = ctx->h_stats->rail;
    return SXGPU_OK;
}

int sxgpu_synth_frames(sxgpu_ctx *ctx, void *d_i2s, uint64_t first_frame, size_t nframes,
                       uint64_t seed, sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    if (nframes == 0)
        return SXGPU_OK;
    if (!d_i2s || reinterpret_cast<uintptr_t>(d_i2s) % 8)
        return ctx->invalid("I2S buffer must be 8-byte aligned");
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    int block = 256;
    uint64_t ctas = (nframes + block - 1) / block;
    int grid = int(std::min<uint64_t>(ctas, uint64_t(ctx->prop.multiProcessorCount) * 8));
    synth_frames_kernel<<<grid, block, 0, st>>>(static_cast<char *>(d_i2s), first_frame, nframes, seed);
    SX_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
    return SXGPU_OK;
}

// ---- plumbing ---------------------------------------------------------------------------
int sxgpu_malloc(sxgpu_ctx *ctx, void **d_ptr, size_t bytes)
{
    if (!ctx || !d_ptr)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaMalloc(d_ptr, bytes));
    return SXGPU_OK;
}
int sxgpu_free(sxgpu_ctx *ctx, void *d_ptr)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaFree(d_ptr));
    return SXGPU_OK;
}
int sxgpu_malloc_host(sxgpu_ctx *ctx, void **h_ptr, size_t bytes)
{
    if (!ctx || !h_ptr)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    NearGpu near(ctx);
    SX_CUDA(ctx, cudaHostAlloc(h_ptr, bytes, cudaHostAllocPortable | cudaHostAllocMapped));
    return SXGPU_OK;
}
int sxgpu_free_host(sxgpu_ctx *ctx, void *h_ptr)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaFreeHost(h_ptr));
    return SXGPU_OK;
}
int sxgpu_host_register(sxgpu_ctx *ctx, void *h_ptr, size_t bytes)
{
    if (!ctx || !h_ptr)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return SXGPU_OK;
}
int sxgpu_host_unregister(sxgpu_ctx *ctx, void *h_ptr)
{
    if (!ctx || !h_ptr)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaHostUnregister(h_ptr));
    return SXGPU_OK;
}
int sxgpu_memcpy_h2d(sxgpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes,
                     sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    SX_CUDA(ctx, cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st));
    ctx->h2d_bytes += bytes;
    return SXGPU_OK;
}
int sxgpu_memcpy_d2h(sxgpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes,
                     sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = call_stream(ctx, stream);
    SX_CUDA(ctx, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
    ctx->d2h_bytes += bytes;
    return SXGPU_OK;
}
int sxgpu_stream_create(sxgpu_ctx *ctx, sxgpu_stream *out)
{
    if (!ctx || !out)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st;
    SX_CUDA(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    *out = st;
    return SXGPU_OK;
}
int sxgpu_stream_destroy(sxgpu_ctx *ctx, sxgpu_stream stream)
{
    if (!ctx || !stream)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaStreamDestroy(static_cast<cudaStream_t>(stream)));
    return SXGPU_OK;
}
int sxgpu_stream_sync(sxgpu_ctx *ctx, sxgpu_stream stream)
{
    if (!ctx)
        return SXGPU_ERR_INVALID;
    SX_CUDA(ctx, cudaSetDevice(ctx->device));
    SX_CUDA(ctx, cudaStreamSynchronize(call_stream(ctx, stream)));
    return SXGPU_OK;
}

int sxgpu_set_option(sxgpu_ctx *ctx, const char *key, int64_t value)
{
    if (!ctx || !key)
        return SXGPU_ERR_INVALID;
    int64_t *slot = option_slot(ctx, key);
    if (!slot)
        return ctx->invalid("unknown option");
    if (value < 0)
        return ctx->invalid("option values are non-negative");
    if (slot == &ctx->numa_node)
        return ctx->invalid("numa_node is read-only");
    std::scoped_lock lock(ctx->lanes[0].mutex, ctx->lanes[1].mutex);
    *slot = value;
    return SXGPU_OK;
}

int sxgpu_get_option(sxgpu_ctx *ctx, const char *key, int64_t *value)
{
    if (!ctx || !key || !value)
        return SXGPU_ERR_INVALID;
    int64_t *slot = option_slot(ctx, key);
    if (!slot)
        return ctx->invalid("unknown option");
    *value = *slot;
    return SXGPU_OK;
}

int sxgpu_get_counter(sxgpu_ctx *ctx, const char *key, uint64_t *value)
{
    if (!ctx || !key || !value)
        return SXGPU_ERR_INVALID;
    if (!std::strcmp(key, "launches")) *value = ctx->launches;
    else if (!std::strcmp(key, "frames_rx")) *value = ctx->frames_rx;
    else if (!std::strcmp(key, "frames_tx")) *value = ctx->frames_tx;
    else if (!std::strcmp(key, "h2d_bytes")) *value = ctx->h2d_bytes;
    else if (!std::strcmp(key, "d2h_bytes")) *value = ctx->d2h_bytes;
    else if (!std::strcmp(key, "resident_launches")) *value = ctx->resident_launches;
    else if (!std::strcmp(key, "resident_calls")) *value = ctx->resident_calls;
    else if (!std::strcmp(key, "flagged_calls")) *value = ctx->flagged_calls;
    else return ctx->invalid("unknown counter");
    return SXGPU_OK;
}

} // extern "C"

// ---------------------------------------------------------------------------------------
// Several GPUs from one process: one context and one host thread per GPU (SURVEY.md section
// 8(e)).  Blocks and streams are independent, so the only thing the GPUs share is the caller's
// list of blocks: block b of a host-buffer list goes to GPU b mod G; a device-buffer block goes to
// the GPU its memory is on.  No data crosses between GPUs and there is no collective.
// ---------------------------------------------------------------------------------------
struct sxgpu_multi {
    std::vector<sxgpu_ctx *> ctx;
    std::unique_ptr<sxhost::WorkerPool> pool; // G - 1 helpers: GPU g is always driven by thread g
    std::mutex mutex;                         // one multi-GPU call at a time
    std::string last_error;
};

namespace {

template <class Op>
int multi_convert_host(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    if (!m)
        return SXGPU_ERR_INVALID;
    if (nblocks == 0)
        return SXGPU_OK;
    if (!blocks)
        return SXGPU_ERR_INVALID;
    std::lock_guard<std::mutex> lock(m->mutex);
    const size_t G = m->ctx.size();
    std::vector<int> rc(G, SXGPU_OK);
    m->pool->run(G, 1, [&](size_t lo, size_t hi) {
        for (size_t g = lo; g < hi; g++) {
            sxgpu_ctx *ctx = m->ctx[g];
            for (uint32_t b = uint32_t(g); b < nblocks && rc[g] == SXGPU_OK; b += uint32_t(G)) {
                rc[g] = convert_host<Op>(ctx, blocks[b].src, 0, blocks[b].dest, 0, size_t(blocks[b].length),
                                         blocks[b].tx_threshold2, lane_of<Op>() ? ctx->tx_variant : ctx->rx_variant);
                if (rc[g] == SXGPU_OK)
                    (lane_of<Op>() ? ctx->frames_tx : ctx->frames_rx) += blocks[b].length;
            }
        }
    });
    for (size_t g = 0; g < G; g++)
        if (rc[g] != SXGPU_OK) {
            m->last_error = "GPU " + std::to_string(m->ctx[g]->device) + ": " + sxgpu_last_error(m->ctx[g]);
            return rc[g];
        }
    return SXGPU_OK;
}

template <class Op>
int multi_convert_batch(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    if (!m)
        return SXGPU_ERR_INVALID;
    if (nblocks == 0)
        return SXGPU_OK;
    if (!blocks)
        return SXGPU_ERR_INVALID;
    std::lock_guard<std::mutex> lock(m->mutex);
    const size_t G = m->ctx.size();
    // Sort the blocks by the GPU their source buffer lives on.
    std::vector<std::vector<sxgpu_block>> mine(G);
    for (uint32_t b = 0; b < nblocks; b++) {
        if (blocks[b].length == 0)
            continue;
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, blocks[b].src) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            m->last_error = "block " + std::to_string(b) + ": source is not device memory";
            return SXGPU_ERR_INVALID;
        }
        size_t g = 0;
        while (g < G && m->ctx[g]->device != attr.device)
            g++;
        if (g == G) {
            m->last_error = "block " + std::to_string(b) + ": its GPU is not part of this group";
            return SXGPU_ERR_INVALID;
        }
        mine[g].push_back(blocks[b]);
    }
    std::vector<int> rc(G, SXGPU_OK);
    m->pool->run(G, 1, [&](size_t lo, size_t hi) {
        for (size_t g = lo; g < hi; g++)
            if (!mine[g].empty())
                rc[g] = convert_batch<Op>(m->ctx[g], mine[g].data(), uint32_t(mine[g].size()), 0, 0, nullptr);
    });
    for (size_t g = 0; g < G; g++)
        if (rc[g] != SXGPU_OK) {
            m->last_error = "GPU " + std::to_string(m->ctx[g]->device) + ": " + sxgpu_last_error(m->ctx[g]);
            return rc[g];
        }
    return SXGPU_OK;
}

} // namespace

extern "C" {

int sxgpu_multi_create(const int *devices, int ndevices, sxgpu_multi **out)
{
    if (!out)
        return SXGPU_ERR_INVALID;
    *out = nullptr;
    if (!devices || ndevices <= 0)
        return SXGPU_ERR_INVALID;
    std::unique_ptr<sxgpu_multi> m(new sxgpu_multi());
    for (int i = 0; i < ndevices; i++) {
        for (int j = 0; j < i; j++)
            if (devices[j] == devices[i]) {
                for (sxgpu_ctx *c : m->ctx)
                    sxgpu_destroy(c);
                return SXGPU_ERR_INVALID; // each GPU once
            }
        sxgpu_ctx *c = nullptr;
        int rc = sxgpu_init(devices[i], &c);
        if (rc != SXGPU_OK) {
            for (sxgpu_ctx *done : m->ctx)
                sxgpu_destroy(done);
            return rc;
        }
        m->ctx.push_back(c);
    }
    m->pool.reset(new sxhost::WorkerPool(unsigned(ndevices - 1)));
    *out = m.release();
    return SXGPU_OK;
}

int sxgpu_multi_destroy(sxgpu_multi *m)
{
    if (!m)
        return SXGPU_ERR_INVALID;
    int worst = SXGPU_OK;
    for (sxgpu_ctx *c : m->ctx) {
        int rc = sxgpu_destroy(c);
        if (rc != SXGPU_OK)
            worst = rc;
    }
    delete m;
    return worst;
}

int sxgpu_multi_size(sxgpu_multi *m) { return m ? int(m->ctx.size()) : 0; }

sxgpu_ctx *sxgpu_multi_context(sxgpu_multi *m, int index)
{
    return (m && index >= 0 && size_t(index) < m->ctx.size()) ? m->ctx[size_t(index)] : nullptr;
}

const char *sxgpu_multi_last_error(sxgpu_multi *m)
{
    static thread_local std::string mine;
    if (!m)
        return "";
    std::lock_guard<std::mutex> lock(m->mutex);
    mine = m->last_error;
    return mine.c_str();
}

int sxgpu_multi_convert_rx_host(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    return multi_convert_host<RxCf32>(m, blocks, nblocks);
}
int sxgpu_multi_convert_tx_host(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    return multi_convert_host<TxCf32>(m, blocks, nblocks);
}
int sxgpu_multi_convert_rx_batch(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    return multi_convert_batch<RxCf32>(m, blocks, nblocks);
}
int sxgpu_multi_convert_tx_batch(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks)
{
    return multi_convert_batch<TxCf32>(m, blocks, nblocks);
}

int sxgpu_multi_sync(sxgpu_multi *m)
{
    if (!m)
        return SXGPU_ERR_INVALID;
    for (sxgpu_ctx *c : m->ctx)
        SX_TRY(sxgpu_stream_sync(c, nullptr));
    return SXGPU_OK;
}

} // extern "C"
