// sx_bank.cuh -- a bank of independent SX1255 stream pairs whose state lives in HBM.
//
// The reference serves one front-end per process and does one readStream + one writeStream
// of a 256-frame period per loop iteration (example/linear_repeater.py:50-71): 2 KiB each way,
// pure latency.  On a B200 the natural unit is thousands of such streams per launch, and then
// the per-stream bookkeeping (SoapySX.cpp:868-1105) is itself data-parallel: every stream
// carries three counters and the rules in host/stream_plan.hpp are pure functions of them.
// So the bank keeps, per stream, in device memory:
//     clock        frames the (virtual) SX1255 has produced/consumed since the streams started
//     rx_position  the RX frame counter (AlsaPcm::position of the capture side, :378)
//     tx_position  the TX frame counter (playback side)
// plus a playback ring of `ring` frames and a capture staging slot of one period, and runs,
// with one warp per stream (up to 8192 streams lane 0 decides and the warp moves the data;
// beyond that the decisions are taken first by thread-per-stream plan kernels, so that no lane
// idles through the timestamp arithmetic):
//     bank_capture_kernel     what readStream decides (bank_plan_read) + stand-in for the I2S
//                             DMA: writes the planned frames into HBM
//     batch_warp_kernel<RxCf32>  the conversion, from the capture slot to the caller's CF32
//     bank_tx_kernel          what writeStream decides (bank_plan_write) + silence for
//                             forwarded-over gaps + the conversion into the playback ring
// and, for the repeater pattern (read, then a timed write of the block just read), all of the
// above in one launch:
//     bank_repeat_warp_kernel<K, IN_REGISTERS, Hook>   K lanes decide for K streams from
//                             registers, then the warp takes each stream through the three
//                             stages back to back: stage by stage through memory (each stage
//                             reading from L2 what the previous one has just written), or with
//                             every intermediate in registers and only the stores (the form
//                             with a hook point, sx_hook.cuh)
//     bank_repeat_kernel      the memory-staged form with a CTA's first warp deciding for 32 streams
// Large banks (bank_is_large: bound by HBM, not by launch latency) run every call -- the fused
// iteration and the separate read and write -- as two kernels instead:
//     bank_plan_{repeat,read,write}_kernel   the decisions, one thread per stream
//     bank_repeat_data_kernel<U, Hook, MODE> the samples: one chunk of vectors per CTA, CTAs handed
//                             out in order by the hardware, every intermediate in registers,
//                             launched as a programmatic dependent of the plan kernel
// and the iteration or a half of it with IIR filters (every bank size) as:
//     bank_plan_{repeat,read,write}_kernel, then bank_repeat_iir_kernel<Hook, MODE>: whole
//                             streams per CTA through shared-memory tiles, as a programmatic
//                             dependent of the plan kernel
// and a half with a FIR filter or resampler (every bank size), with or without an oscillator
// mixing the full-rate frames (digital down- and up-conversion), as:
//     bank_plan_{read,write}_kernel, then bank_fir_kernel<R, MODE, Nco>: fir_apply_kernel's
//                             polyphase tiles with the frames taken from the capture or stored
//                             into the ring, as a programmatic dependent of the plan kernel, then
//                             bank_fir_read_tail_kernel<Nco> / fir_history_kernel<Nco>, which also
//                             advance the phases when Nco is NcoView
// The virtual clock follows the same rule as the host-side ALSA stand-in: it moves when a
// blocking transfer must wait (by exactly the deficit) or when the owner advances it.
#pragma once

#include "host/stream_plan.hpp"
#include "sx_fir.cuh"
#include "sx_iir.cuh"
#include "sx_kernels.cuh"
#include "sx_nco.cuh"
#include "sx_time.h"

namespace sx {

// Programmatic dependent launch (no-ops in a kernel that was launched the ordinary way): the
// first lets the next kernel of the stream be set up on the SMs while this one is still running;
// the second, in that next kernel, waits until this one has finished and its stores are visible.
__device__ __forceinline__ void pdl_launch_dependents()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

struct BankState {
    uint32_t nstreams;
    uint32_t period;
    uint64_t ring; // playback/capture ring size in frames (sxplan::Geometry::buffer)
    double sample_rate;
    float thr2;
    uint64_t seed;

    long long *clock;
    long long *rx_position;
    long long *tx_position;

    // results of the last read / write, per stream
    int *rx_ret;
    int *rx_flags;
    long long *rx_time_ns;
    int *tx_ret;

    // plans handed from the plan kernels to the data kernels
    long long *rx_first_frame; // counter value of the first frame of the block being read
    BlockDesc *rx_blocks;      // staging slot -> caller's CF32 block
    long long *tx_write_position;
    long long *tx_gap_start; // forwarded-over region to be silenced
    long long *tx_gap_length;
    long long *tx_ring_offset; // the block's place in playback_ring, see bank_ring_offset(); written by the
                               // plan kernels for the data kernels

    char *capture_stage; // [nstreams][period] I2S frames
    char *playback_ring; // [ring / period][nstreams][period] I2S frames, see ring_frame()
};

// Where frame `pos` of stream s's playback ring lives.  Each stream has a ring of `ring` frames
// (a whole number of periods), but the rings are stored time-major: period-long slice
// (pos / period) mod (ring / period) of EVERY stream is contiguous.  Streams that run in
// lock-step -- the normal case: one sample clock -- then write one dense region per iteration
// (nstreams x period x 8 bytes) instead of nstreams regions ring x 8 bytes apart, which at
// 65536 streams meant one 2 KiB write per 512 KiB of a 32 GiB arena: a TLB miss and a DRAM row
// per write.  A block that does not start on a period boundary spans two slices.
__device__ __forceinline__ char *ring_frame(const BankState &b, uint64_t s, uint64_t pos)
{
    const uint32_t P = b.period;
    if ((P & (P - 1)) == 0) { // a power of two (the default 256 is): so is the ring, 65536, and everything is a shift
        const uint32_t lg = 31 - __clz(P);
        const uint64_t slice = (pos >> lg) & ((b.ring >> lg) - 1);
        return b.playback_ring + ((((slice * b.nstreams + s) << lg) + (pos & (P - 1))) << 3);
    }
    const uint64_t slice = (pos / b.period) % (b.ring / b.period);
    return b.playback_ring + ((slice * b.nstreams + s) * b.period + pos % b.period) * 8;
}

// What the data kernels find in tx_ring_offset[s] for a block written at counter `at`: the byte
// offset in playback_ring of its first frame (a multiple of 8), + 1 when the block does not start
// on a period boundary of the ring (it then spans two slices); -1 when it was discarded as late.
__device__ __forceinline__ long long bank_ring_offset(const BankState &b, uint64_t s, long long at)
{
    return at >= 0 ? (long long)(ring_frame(b, s, uint64_t(at)) - b.playback_ring) + (uint64_t(at) % b.period != 0 ? 1 : 0)
                   : -1;
}

// Two converted frames, at and at + 1, into stream s's ring one by one: the store of a block that
// straddles two slices of the time-major ring (rare: a stream out of step).
__device__ __forceinline__ void ring_store_pair(const BankState &b, uint64_t s, uint64_t at, const Pack<4> &out)
{
    Pack<2> f0, f1;
    f0.w[0] = out.w[0], f0.w[1] = out.w[1], f1.w[0] = out.w[2], f1.w[1] = out.w[3];
    st_stream<8>(ring_frame(b, s, at), f0);
    st_stream<8>(ring_frame(b, s, at + 1), f1);
}

// The stand-in I2S DMA: capture frame k of the stream whose generator is seeded with `seed`
// (the bank's seed + the stream's index) as one I2S frame, and frames k, k + 1 as one vector.
__device__ __forceinline__ Pack<2> capture_frame(uint64_t seed, uint64_t k)
{
    const uint64_t z = sx_synth_frame(seed, k);
    Pack<2> p;
    p.w[0] = uint32_t(z);
    p.w[1] = uint32_t(z >> 32);
    return p;
}
__device__ __forceinline__ Pack<4> capture_pair(uint64_t seed, uint64_t k)
{
    const uint64_t z0 = sx_synth_frame(seed, k), z1 = sx_synth_frame(seed, k + 1);
    Pack<4> p;
    p.w[0] = uint32_t(z0), p.w[1] = uint32_t(z0 >> 32);
    p.w[2] = uint32_t(z1), p.w[3] = uint32_t(z1 >> 32);
    return p;
}

// Silence for frames [start, start + n) of stream s's ring, written by the lanes of a warp side by side.
__device__ __forceinline__ void ring_zero(const BankState &b, uint64_t s, long long start, long long n, uint32_t lane)
{
    Pack<2> zero;
    zero.w[0] = zero.w[1] = 0;
    for (long long i = lane; i < n; i += 32)
        st_stream<8>(ring_frame(b, s, uint64_t(start + i)), zero);
}

// A forwarded-over region [start, start + gap) older than one lap: only its last lap is still in the ring.
__device__ __forceinline__ void clamp_gap_to_ring(const BankState &b, long long &start, long long &gap)
{
    if (gap > (long long)b.ring) {
        start += gap - (long long)b.ring;
        gap = (long long)b.ring;
    }
}

// ALSA plays zeros for regions the application skipped (silence_size = boundary, :493-496): the
// warp silences stream s's forwarded-over region [start, start + gap) before the block is written.
// A gap of a whole lap or more silences the slots the block is about to take, hence the barrier.
__device__ __forceinline__ void bank_silence_gap(const BankState &b, uint64_t s, long long start, long long gap, uint32_t lane)
{
    clamp_gap_to_ring(b, start, gap);
    ring_zero(b, s, start, gap, lane);
    __syncwarp();
}

constexpr int SX_HAS_TIME = 1 << 2; // SOAPY_SDR_HAS_TIME

// From here up a bank's iteration is bound by HBM, not by launch latency, and runs as a plan
// kernel plus a data kernel of hardware-scheduled CTAs (measured crossover: equal at 4096 x 256
// frames, 10 % ahead at 16384 x 256, 13 % at 65536 x 256; profiles/r02_summary.md section 5).
inline bool bank_is_large(const BankState &b)
{
    return b.nstreams >= 16384 && uint64_t(b.nstreams) * b.period >= (uint64_t(1) << 21) && b.period % 2 == 0 && b.period >= 4;
}

// readStream(stream, buf, period, timeoutUs > 0) for stream s: SoapySX.cpp:897-959.
// Run by one lane of the warp that owns the stream.  The counters come in as values and the
// decisions go out as values (and to the state arrays), so that a caller which goes on to plan
// the write of the same stream does not wait for its own stores to come back from memory.
struct BankReadPlan {
    long long first;   // counter value of the first frame of the block
    long long time_ns; // its timestamp
    long long clock;   // the stream's clock after the read
};

__device__ __forceinline__ BankReadPlan bank_plan_read_core(const BankState &b, uint64_t s, char *cf32_out,
                                                            long long clock, long long pos)
{
    const sxplan::Geometry geo = {b.period, b.ring};
    long pending = long(clock - pos);

    unsigned long skip = sxplan::overrun_skip(pending, geo); // :910-915
    if (skip) {
        long moved = long(skip) < pending ? long(skip) : pending; // forward() moves at most what is pending
        pos += moved;
        pending -= moved;
    }
    const long length = long(b.period);
    if (pending < length) // a blocking read waits for the I2S clock
        clock += length - pending;

    BankReadPlan plan;
    plan.first = pos;
    plan.time_ns = sx_ticks_to_time_ns(pos, b.sample_rate); // timestamp of the first frame (:950)
    plan.clock = clock;
    b.rx_time_ns[s] = plan.time_ns;
    b.rx_flags[s] = SX_HAS_TIME;
    b.rx_first_frame[s] = pos;
    b.rx_ret[s] = int(length);
    b.rx_position[s] = pos + length;
    b.clock[s] = clock;

    BlockDesc d;
    d.src = b.capture_stage + size_t(s) * b.period * 8;
    d.dst = cf32_out + size_t(s) * b.period * 8;
    d.length = uint64_t(length);
    d.thr2 = 0.0f;
    d.reserved = 0;
    b.rx_blocks[s] = d;
    return plan;
}

__device__ __forceinline__ BankReadPlan bank_plan_read(const BankState &b, uint64_t s, char *cf32_out)
{
    return bank_plan_read_core(b, s, cf32_out, b.clock[s], b.rx_position[s]);
}

// One warp per stream: lane 0 makes readStream's decisions, then the warp plays the I2S DMA --
// frame k of stream s is sx_synth_frame(seed + s, k) -- and writes the planned frames into the
// stream's capture slot.  The conversion itself is a separate launch (batch_warp_kernel<RxCf32>
// over the descriptors written here): it reads the frames back from HBM as it would after a
// real DMA.
// `fused`: lane 0 plans here (few streams: saves a launch).  Otherwise bank_plan_read_kernel
// has already planned every stream with one thread each (many streams: keeps all lanes busy).
__global__ void bank_plan_read_kernel(BankState b, char *cf32_out)
{
    pdl_launch_dependents(); // a data kernel launched as our programmatic dependent may set itself up now
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < b.nstreams)
        bank_plan_read(b, s, cf32_out);
}

__global__ void bank_capture_kernel(BankState b, char *cf32_out, bool fused, bool synth)
{
    const uint32_t lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * warps_per_cta;
    for (uint64_t s = uint64_t(blockIdx.x) * warps_per_cta + (threadIdx.x >> 5); s < b.nstreams; s += nwarps) {
        long long first_ll = 0;
        if (lane == 0) {
            first_ll = fused ? bank_plan_read(b, s, cf32_out).first : b.rx_first_frame[s];
        }
        const uint64_t first = uint64_t(__shfl_sync(0xffffffffu, first_ll, 0));
        if (!synth) // the slot was filled from outside (sxgpu_bank_ingest)
            continue;
        char *out = b.capture_stage + s * b.period * 8;
        for (uint32_t i = lane; i < b.period; i += 32) {
            const Pack<2> p = capture_frame(b.seed + s, first + i);
            st_stream<8>(out + size_t(i) * 8, p);
        }
    }
}

// writeStream(stream, buf, period, flags, timeNs, timeoutUs > 0) for stream s: :989-1097.
// Run by one lane of the stream's warp; counters in and decisions out as values, as above.
struct BankWritePlan {
    long long at;    // counter value the block is written at, -1: discarded as late
    long long gap;   // length of the forwarded-over region to be silenced
    long long start; // where that region starts
};

__device__ __forceinline__ BankWritePlan bank_plan_write_core(const BankState &b, uint64_t s, bool timed,
                                                              long long time_ns, long long clock, long long pos)
{
    const long long ring = (long long)b.ring, period = (long long)b.period;
    const long queued = long(pos - clock); // ALSA delay: written but not yet played

    const long long ticks = timed ? sx_time_ns_to_ticks(time_ns, b.sample_rate) : 0;
    sxplan::TxPlacement where = sxplan::place_tx_block(pos, queued, timed, ticks, b.period);

    BankWritePlan plan = {-1, 0, pos};
    if (where.discard) { // :1017-1023: report written, write nothing
        b.tx_gap_start[s] = pos;
        b.tx_gap_length[s] = 0;
        b.tx_ret[s] = int(period);
        b.tx_write_position[s] = -1;
        return plan;
    }

    // :1043-1073: forward the write pointer to the block's position, waiting for ring space --
    // in closed form (sxplan::clock_after_forward), so that a far-future or garbage timestamp
    // costs the same few instructions as any other instead of one loop turn per period of gap.
    const long long gap = where.write_position - pos;
    if (gap > 0) {
        plan.gap = gap;
        clock = sxplan::clock_after_forward(clock, pos, where.write_position, ring, period);
        pos = where.write_position;
    }

    // blocking snd_pcm_writei of one period (:1093)
    long long room = clock + ring - pos;
    if (room < period)
        clock += period - room;

    plan.at = pos;
    b.tx_gap_start[s] = plan.start;
    b.tx_gap_length[s] = plan.gap;
    b.tx_write_position[s] = pos;
    b.tx_ret[s] = int(period);
    b.tx_position[s] = pos + period;
    b.clock[s] = clock;
    return plan;
}

// time_ns == nullptr means "the timestamp of this stream's last read plus rx_time_offset_ns",
// the repeater pattern (example/linear_repeater.py:64-69).
__device__ __forceinline__ BankWritePlan bank_plan_write(const BankState &b, uint64_t s, int flags,
                                                         const long long *time_ns, long long rx_time_offset_ns)
{
    const bool timed = (flags & SX_HAS_TIME) != 0;
    long long t = 0;
    if (timed)
        t = time_ns ? time_ns[s] : b.rx_time_ns[s] + rx_time_offset_ns;
    return bank_plan_write_core(b, s, timed, t, b.clock[s], b.tx_position[s]);
}

// readStream then writeStream(HAS_TIME, that read's timestamp + rx_time_offset_ns) of one stream:
// the three counters are loaded side by side, and the write is planned from the read's results
// without a trip through memory.  Same stores, in the same order, as the two separate plans.
__device__ __forceinline__ void bank_plan_repeat(const BankState &b, uint64_t s, char *cf32, long long rx_time_offset_ns,
                                                 long long &first, BankWritePlan &w)
{
    const long long clock = b.clock[s], rx_pos = b.rx_position[s], tx_pos = b.tx_position[s];
    const BankReadPlan r = bank_plan_read_core(b, s, cf32, clock, rx_pos);
    w = bank_plan_write_core(b, s, true, r.time_ns + rx_time_offset_ns, r.clock, tx_pos);
    first = r.first;
}

// The data side of writeStream for stream s, done by one warp: silence for the forwarded-over
// region [start, start + gap), then the block converted into the playback ring at counter `at`
// (at < 0: the block was discarded as late, nothing is written).
__device__ __forceinline__ void bank_play_block(const BankState &b, uint64_t s, const char *cf32_in, long long at,
                                                long long gap, long long start, uint32_t lane)
{
    if (at < 0)
        return;
    if (gap > 0)
        bank_silence_gap(b, s, start, gap, lane);

    // The block may straddle a period boundary of the ring: at most two contiguous spans.
    const uint64_t into = uint64_t(at) % b.period;
    const uint64_t first_span = into ? b.period - into : b.period;
    BlockDesc d;
    d.thr2 = b.thr2;
    d.reserved = 0;
    d.src = cf32_in + s * b.period * 8;
    d.dst = ring_frame(b, s, uint64_t(at));
    d.length = first_span;
    convert_span<TxCf32>(d, 0, first_span, lane, 32);
    if (first_span < b.period) {
        d.src = cf32_in + (s * b.period + first_span) * 8;
        d.dst = ring_frame(b, s, uint64_t(at) + first_span);
        d.length = b.period - first_span;
        convert_span<TxCf32>(d, 0, d.length, lane, 32);
    }
}

// Silence for the forwarded-over regions of a warp's 32 streams (ALSA plays zeros for what the
// application skipped, :493-496), written by the whole warp stream after stream: 32 frames per
// store instruction, side by side, instead of one thread per stream walking its gap alone.  Every
// lane of the warp must call this (lanes without a stream or without a gap pass gap = 0).
__device__ __forceinline__ void bank_silence_by_warp(const BankState &b, uint64_t s, long long start, long long gap)
{
    const uint32_t lane = threadIdx.x & 31;
    clamp_gap_to_ring(b, start, gap);
    unsigned pending = __ballot_sync(0xffffffffu, gap > 0);
    while (pending) {
        const int j = __ffs(pending) - 1;
        pending &= pending - 1;
        const uint64_t sj = __shfl_sync(0xffffffffu, s, j);
        const long long start_j = __shfl_sync(0xffffffffu, start, j), gap_j = __shfl_sync(0xffffffffu, gap, j);
        ring_zero(b, sj, start_j, gap_j, lane);
    }
}

// `for_data_kernel`: the samples follow in bank_repeat_data_kernel<..., kBankModeWrite>, which wants
// the block's place in the ring as a byte offset and the silence of a forwarded-over gap already
// written (bank_tx_kernel, the warp-per-stream data side, does both itself).
__global__ void bank_plan_write_kernel(BankState b, int flags, const long long *time_ns,
                                       long long rx_time_offset_ns, bool for_data_kernel)
{
    pdl_launch_dependents();
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    BankWritePlan w = {-1, 0, 0};
    if (s < b.nstreams) {
        w = bank_plan_write(b, s, flags, time_ns, rx_time_offset_ns);
        if (for_data_kernel)
            b.tx_ring_offset[s] = bank_ring_offset(b, s, w.at);
    }
    if (for_data_kernel) // (uniform over the grid: every lane gets here)
        bank_silence_by_warp(b, s, w.start, (s < b.nstreams && w.at >= 0) ? w.gap : 0);
}

// One warp per stream: lane 0 makes writeStream's decisions, then the warp writes silence for
// the forwarded-over region and converts the block into the stream's playback ring.
__global__ void bank_tx_kernel(BankState b, const char *cf32_in, int flags, const long long *time_ns,
                               long long rx_time_offset_ns, bool fused)
{
    const uint32_t lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * warps_per_cta;
    for (uint64_t s = uint64_t(blockIdx.x) * warps_per_cta + (threadIdx.x >> 5); s < b.nstreams; s += nwarps) {
        long long at = 0, gap = 0, start = 0;
        if (lane == 0) {
            if (fused) { // decisions straight from the plan, not back through memory
                const BankWritePlan w = bank_plan_write(b, s, flags, time_ns, rx_time_offset_ns);
                at = w.at;
                gap = w.gap;
                start = w.start;
            } else {
                at = b.tx_write_position[s];
                gap = b.tx_gap_length[s];
                start = b.tx_gap_start[s];
            }
        }
        at = __shfl_sync(0xffffffffu, at, 0);
        gap = __shfl_sync(0xffffffffu, gap, 0);
        start = __shfl_sync(0xffffffffu, start, 0);
        bank_play_block(b, s, cf32_in, at, gap, start, lane);
    }
}

// One stream's share of the repeater iteration, done by one warp once the decisions are taken:
// the stand-in DMA writes the planned frames into the capture slot, the RX conversion reads
// them back (as it would after a real DMA) into the caller's CF32 block, and the TX conversion
// reads that block into the playback ring.
__device__ __forceinline__ void bank_repeat_stream(const BankState &b, uint64_t s, char *cf32, uint64_t first,
                                                   long long at, long long gap, long long start, uint32_t lane,
                                                   bool capture_in_slot)
{
    char *slot = b.capture_stage + s * b.period * 8;
    for (uint32_t i = lane; i < b.period && !capture_in_slot; i += 32) {
        const Pack<2> p = capture_frame(b.seed + s, first + i);
        st_stream<8>(slot + size_t(i) * 8, p);
    }
    __syncwarp(); // the slot is complete before any lane reads it back
    BlockDesc d;
    d.src = slot;
    d.dst = cf32 + s * b.period * 8;
    d.length = b.period;
    d.thr2 = 0.0f;
    d.reserved = 0;
    convert_span<RxCf32>(d, 0, d.length, lane, 32);
    __syncwarp(); // the CF32 block is complete before the TX stage reads it
    bank_play_block(b, s, cf32, at, gap, start, lane);
}

// The same share with every intermediate kept in registers: a lane owns 16-byte vectors
// v = lane, lane + 32, ... of the period (two frames each), produces their capture frames,
// converts them to CF32 and on to I2S words without a trip through memory, and issues the three
// stores -- capture slot, caller's CF32 block, playback ring -- back to back.  Nothing is read
// back, so a stream costs its plan's one round trip (the three counters) and then only stores.
// `capture_in_slot`: the capture slot was filled from outside (sxgpu_bank_ingest); it is read
// (one round trip, all vectors in flight at once) instead of being produced here.
// Needs an even period and 16-byte aligned CF32 blocks; a block that does not start on a period
// boundary of the ring falls back to frame-wide stores for the ring side.
template <class Hook>
__device__ __forceinline__ void bank_repeat_stream_reg(const BankState &b, uint64_t s, char *cf32, uint64_t first,
                                                       long long at, long long gap, long long start, uint32_t lane,
                                                       bool capture_in_slot, const Hook &hook)
{
    constexpr int U = 4; // 16-byte vectors a lane has in flight: a 256-frame period in one go
    char *slot = b.capture_stage + s * b.period * 8;
    char *cf = cf32 + s * b.period * 8;
    const uint32_t nvec = b.period / 2;

    if (at >= 0 && gap > 0) // rare: late start, underrun
        bank_silence_gap(b, s, start, gap, lane);
    // Streams in lock-step write whole period slices of the ring: 16-byte stores.  A block that
    // starts inside a slice goes frame by frame.
    const bool ring_vec = at >= 0 && uint64_t(at) % b.period == 0;
    char *ring = ring_vec ? ring_frame(b, s, uint64_t(at)) : nullptr;

    for (uint32_t base = 0; base < nvec; base += 32 * U) {
        Pack<4> cap[U], mid[U], out[U];
        if (capture_in_slot) {
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t v = base + lane + 32 * u;
                if (v < nvec)
                    cap[u] = ld_stream<16>(slot + size_t(v) * 16);
            }
        } else {
#pragma unroll
            for (int u = 0; u < U; u++)
                cap[u] = capture_pair(b.seed + s, first + 2 * uint64_t(base + lane + 32 * u));
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            RxCf32::apply<2>(cap[u], mid[u], 0.0f);
            if (base + lane + 32 * u < nvec)
                hook(mid[u], s, 2 * (base + lane + 32 * u)); // user DSP between RX and TX, identity by default
            TxCf32::apply<2>(mid[u], out[u], b.thr2);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint32_t v = base + lane + 32 * u;
            if (v >= nvec)
                continue;
            if (!capture_in_slot)
                st_stream<16>(slot + size_t(v) * 16, cap[u]);
            st_stream<16>(cf + size_t(v) * 16, mid[u]);
            if (ring_vec)
                st_stream<16>(ring + size_t(v) * 16, out[u]);
            else if (at >= 0)
                ring_store_pair(b, s, uint64_t(at) + 2 * uint64_t(v), out[u]);
        }
    }
}

// The hook the fused iteration applies to each pair of CF32 samples between the RX and the TX
// conversion.  Identity here; csrc/sx_hook.cuh has the interface and an example.
struct IdentityHook {
    __device__ __forceinline__ void operator()(Pack<4> &, uint64_t, uint32_t) const {}
};

// The repeater iteration in one launch: readStream(period) on every stream, then
// writeStream(period, HAS_TIME, that read's timestamp + rx_time_offset_ns) of the block just
// read (example/linear_repeater.py:50-71 without the filters).  State and results are exactly
// those of bank_read followed by bank_write; what changes is the schedule.  A CTA takes 32
// streams at a time: its first warp takes the 32 streams' decisions, one stream per lane, and
// hands them over in shared memory; then each warp carries its streams through all three
// stages -- stand-in DMA into the capture slot, RX conversion into the caller's CF32 block, TX
// conversion into the playback ring -- so each stage reads what the previous one has just
// written while it is still in L2, and only the three writes (24 B/frame) reach HBM instead of
// 40 B/frame over five launches.
constexpr int kRepeatGroup = 32;

__global__ void __launch_bounds__(256) bank_repeat_kernel(BankState b, char *cf32, long long rx_time_offset_ns,
                                                          bool capture_in_slot)
{
    __shared__ long long s_first[kRepeatGroup], s_at[kRepeatGroup], s_gap[kRepeatGroup], s_start[kRepeatGroup];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps_per_cta = blockDim.x >> 5;
    const uint64_t ngroups = (uint64_t(b.nstreams) + kRepeatGroup - 1) / kRepeatGroup;
    for (uint64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const uint64_t base = g * kRepeatGroup;
        const uint32_t count = uint32_t(b.nstreams - base < kRepeatGroup ? b.nstreams - base : kRepeatGroup);
        if (threadIdx.x < count) {
            const uint64_t s = base + threadIdx.x;
            long long first;
            BankWritePlan w;
            bank_plan_repeat(b, s, cf32, rx_time_offset_ns, first, w);
            s_first[threadIdx.x] = first;
            s_at[threadIdx.x] = w.at;
            s_gap[threadIdx.x] = w.gap;
            s_start[threadIdx.x] = w.start;
        }
        __syncthreads();
        for (uint32_t j = warp; j < count; j += warps_per_cta) {
            const uint64_t s = base + j;
            bank_repeat_stream(b, s, cf32, uint64_t(s_first[j]), s_at[j], s_gap[j], s_start[j], lane, capture_in_slot);
        }
        __syncthreads(); // the next group's plans overwrite the shared arrays
    }
}

// The same iteration with every warp on its own: a warp takes K consecutive streams at a time,
// lanes 0..K-1 take their decisions, and the warp then carries them through the three stages.
// No shared memory, no CTA barrier, and K sets the granularity: small K spreads S streams more
// evenly over the resident warps, large K spends fewer issue slots on the (one-lane-per-stream)
// decisions.  IN_REGISTERS: each stream's stages keep their intermediates in registers and only
// store (bank_repeat_stream_reg, the form with a hook point: even periods and 16-byte aligned
// CF32 only); otherwise they go through memory stage by stage (bank_repeat_stream, no hook).
template <int K, bool IN_REGISTERS = false, class Hook = IdentityHook>
__global__ void __launch_bounds__(256) bank_repeat_warp_kernel(BankState b, char *cf32, long long rx_time_offset_ns,
                                                               bool capture_in_slot, Hook hook)
{
    const uint32_t lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * warps_per_cta;
    const uint64_t nchunks = (uint64_t(b.nstreams) + K - 1) / K;
    for (uint64_t c = uint64_t(blockIdx.x) * warps_per_cta + (threadIdx.x >> 5); c < nchunks; c += nwarps) {
        const uint64_t base = c * K;
        const uint32_t count = uint32_t(b.nstreams - base < K ? b.nstreams - base : K);
        long long my_first = 0, my_at = -1, my_gap = 0, my_start = 0;
        if (lane < count) {
            BankWritePlan w;
            bank_plan_repeat(b, base + lane, cf32, rx_time_offset_ns, my_first, w);
            my_at = w.at;
            my_gap = w.gap;
            my_start = w.start;
        }
#pragma unroll
        for (uint32_t j = 0; j < K; j++) {
            const uint64_t first = uint64_t(__shfl_sync(0xffffffffu, my_first, j));
            const long long at = __shfl_sync(0xffffffffu, my_at, j);
            const long long gap = __shfl_sync(0xffffffffu, my_gap, j);
            const long long start = __shfl_sync(0xffffffffu, my_start, j);
            if (j >= count) // count is the same in every lane
                break;
            if constexpr (IN_REGISTERS)
                bank_repeat_stream_reg(b, base + j, cf32, first, at, gap, start, lane, capture_in_slot, hook);
            else
                bank_repeat_stream(b, base + j, cf32, first, at, gap, start, lane, capture_in_slot);
        }
    }
}

// The last `nframes` frames each stream wrote (ending at its TX counter), copied out of the
// playback rings into dst[stream - first_stream][nframes]: what the I2S DMA would fetch next.
// One warp per stream; dst is device memory or device-mapped pinned host memory.
__global__ void bank_drain_kernel(BankState b, uint32_t first_stream, uint32_t count, uint32_t nframes, char *dst)
{
    const uint32_t lane = threadIdx.x & 31, warps_per_cta = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * warps_per_cta;
    for (uint64_t j = uint64_t(blockIdx.x) * warps_per_cta + (threadIdx.x >> 5); j < count; j += nwarps) {
        const uint64_t s = first_stream + j;
        const long long end = b.tx_position[s];
        char *out = dst + j * uint64_t(nframes) * 8;
        for (uint32_t i = lane; i < nframes; i += 32) {
            const long long p = end - (long long)nframes + i;
            Pack<2> f;
            f.w[0] = f.w[1] = 0; // before the stream's first frame: silence
            if (p >= 0)
                f = ld_stream<8>(ring_frame(b, s, uint64_t(p)));
            st_stream<8>(out + size_t(i) * 8, f);
        }
    }
}

// nframes frames of ONE stream's ring starting at counter value `position`, gathered into a
// contiguous buffer (sxgpu_bank_playback: tests and inspection, not a data path).
__global__ void bank_gather_kernel(BankState b, uint32_t stream, long long position, uint64_t nframes, char *dst)
{
    for (uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nframes; i += uint64_t(gridDim.x) * blockDim.x)
        st_stream<8>(dst + i * 8, ld_stream<8>(ring_frame(b, stream, uint64_t(position) + i)));
}

// ---------------------------------------------------------------------------------------
// The repeater iteration as two launches: decisions, then data.
//
// bank_plan_repeat_kernel: one thread per stream takes readStream's and the timed
// writeStream's decisions (bank_plan_repeat: same stores, same order as every other schedule),
// leaves the block's place in the ring as a byte offset for the data kernel and, warp by warp,
// writes the silence of forwarded-over gaps -- rare, and off the data kernel's path.
// The data kernel is bank_repeat_data_kernel, further down.  (A data kernel on the bulk-async
// schedule of round 1 -- persistent CTAs, 2048-frame tiles through shared memory, bulk stores --
// was measured at 125 us for 65536 streams against 61 and is gone: commit 354f3f1 has it.)
// ---------------------------------------------------------------------------------------
__global__ void bank_plan_repeat_kernel(BankState b, char *cf32, long long rx_time_offset_ns)
{
    pdl_launch_dependents(); // the data kernel may take its place on the SMs now; it waits for us before it reads
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    BankWritePlan w = {-1, 0, 0};
    if (s < b.nstreams) {
        long long first;
        bank_plan_repeat(b, s, cf32, rx_time_offset_ns, first, w);
        b.tx_ring_offset[s] = bank_ring_offset(b, s, w.at);
    }
    bank_silence_by_warp(b, s, w.start, (s < b.nstreams && w.at >= 0) ? w.gap : 0);
}

// ---------------------------------------------------------------------------------------
// The data side: hardware-scheduled CTAs.
//
// Every one-launch schedule above runs a persistent grid, and every one of them -- memory-staged,
// register-resident -- lands within a few percent of what *plain stores of the same bytes from a
// persistent grid* reach (tools/experiments/bank_limits.cu: 65.6 us for the 402 MB of 65536
// streams x 256 frames, exactly cudaMemset's time over the same three regions).  The same bytes
// written by CTAs that each take one chunk and leave -- handed out in index order by the hardware,
// so that the addresses in flight form one compact window moving through each region -- take
// 56-58 us, arithmetic included.  The streams' periods lie side by side in the capture slots and
// in the caller's CF32 buffer, so those two are flat arrays; the ring side is flat too whenever a
// block starts on a period boundary of the ring (frame-wide stores otherwise).
// ---------------------------------------------------------------------------------------
// The decisions are taken beforehand by bank_plan_repeat_kernel (one thread per stream, every
// stream of the bank side by side): they are a chain of dependent 64-bit divisions and
// double-precision operations, a few microseconds of latency per stream however few lanes run it,
// so taken inside the data CTAs they hold a whole CTA's registers and threads idle for longer than
// its stores take (that one-launch form was measured at 75.8 us against 61.3 and is gone: commit
// 354f3f1 has it as bank_repeat_direct_kernel).  CTA c takes vectors [c * 256 * U, (c + 1) * 256 * U) of the flat
// capture and CF32 arrays; its first threads fetch the streams' first-frame counters and ring
// offsets into shared memory while the others already have the capture loads in flight.
// MODE: the whole iteration, or one half of it for the separate calls (sxgpu_bank_read: capture
// and RX conversion, 16 B/frame written, or 8 read + 8 written with ingested capture;
// sxgpu_bank_write: the CF32 block loaded, TX conversion, 8 read + 8 written).
constexpr int kBankModeRepeat = 0, kBankModeRead = 1, kBankModeWrite = 2;

template <int U, class Hook, int MODE = kBankModeRepeat>
__global__ void __launch_bounds__(256) bank_repeat_data_kernel(BankState b, char *cf32, bool capture_in_slot, Hook hook)
{
    // streams a CTA can touch: 256 * U vectors of at least two vectors per stream (period >= 4,
    // checked by the host), plus one for a chunk that starts inside a stream
    constexpr int kMaxStreams = 256 * U / 2 + 1;
    __shared__ long long s_first[kMaxStreams], s_off[kMaxStreams];

    const uint32_t nvec = b.period / 2;
    const uint64_t total = uint64_t(b.nstreams) * nvec;
    const uint64_t v0 = uint64_t(blockIdx.x) * (256 * U);
    if (v0 >= total)
        return;
    const bool pow2 = (nvec & (nvec - 1)) == 0;
    const uint32_t log2v = 31 - __clz(nvec);
    const uint64_t s0 = pow2 ? v0 >> log2v : v0 / nvec;                       // first stream this CTA touches
    const uint64_t vlast = v0 + 256 * U - 1 < total - 1 ? v0 + 256 * U - 1 : total - 1;
    const uint32_t count = uint32_t((pow2 ? vlast >> log2v : vlast / nvec) - s0) + 1; // <= 256 * U / nvec + 1
    pdl_wait(); // the decisions (and, before them, the previous iteration's samples) are in memory
    for (uint32_t j = threadIdx.x; j < count; j += 256) {
        if (MODE != kBankModeWrite)
            s_first[j] = b.rx_first_frame[s0 + j];
        if (MODE != kBankModeRead)
            s_off[j] = b.tx_ring_offset[s0 + j];
    }
    Pack<4> cap[U], mid[U], out[U];
    if (MODE == kBankModeWrite) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = v0 + u * 256 + threadIdx.x;
            if (v < total)
                mid[u] = ld_stream<16>(cf32 + v * 16);
        }
    } else if (capture_in_slot) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = v0 + u * 256 + threadIdx.x;
            if (v < total)
                cap[u] = ld_stream<16>(b.capture_stage + v * 16);
        }
    }
    __syncthreads();

    // Which stream (relative to s0) a vector belongs to and where in its period, in 32-bit
    // arithmetic: the CTA's vectors start r0 vectors into stream s0.
    const uint32_t r0 = uint32_t(v0 - s0 * nvec);
    uint32_t jj[U], kk[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint32_t local = r0 + u * 256 + threadIdx.x;
        const uint32_t j = pow2 ? local >> log2v : local / nvec;
        jj[u] = v0 + u * 256 + threadIdx.x < total ? j : 0;
        kk[u] = pow2 ? local & (nvec - 1) : local - j * nvec;
        if (MODE != kBankModeWrite && !capture_in_slot)
            cap[u] = capture_pair(b.seed + s0 + jj[u], uint64_t(s_first[jj[u]]) + 2 * uint64_t(kk[u]));
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint64_t v = v0 + u * 256 + threadIdx.x;
        if (MODE != kBankModeWrite)
            RxCf32::apply<2>(cap[u], mid[u], 0.0f);
        if (MODE == kBankModeRepeat && v < total)
            hook(mid[u], s0 + jj[u], 2 * kk[u]); // user DSP between RX and TX, identity by default
        if (MODE != kBankModeRead)
            TxCf32::apply<2>(mid[u], out[u], b.thr2);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint64_t v = v0 + u * 256 + threadIdx.x;
        if (v >= total)
            continue;
        if (MODE != kBankModeWrite) {
            if (!capture_in_slot)
                st_stream<16>(b.capture_stage + v * 16, cap[u]);
            st_stream<16>(cf32 + v * 16, mid[u]);
        }
        if (MODE == kBankModeRead)
            continue;
        const long long off = s_off[jj[u]];
        if (off < 0)
            continue; // discarded as late
        if ((off & 1) == 0) {
            // the block starts on a period boundary of the ring: one contiguous, 16-byte aligned span
            st_stream<16>(b.playback_ring + off + size_t(kk[u]) * 16, out[u]);
        } else {
            // it straddles two slices of the time-major ring: frame by frame
            ring_store_pair(b, s0 + jj[u], uint64_t(b.tx_write_position[s0 + jj[u]]) + 2 * uint64_t(kk[u]), out[u]);
        }
    }
}

// ---------------------------------------------------------------------------------------
// The repeater iteration with its filters (sxgpu_bank_repeat_filtered, sx_hook.cuh): read, pre
// cascade, the hook, post cascade, then the CF32 block and the timed write.  Same state, results,
// CF32 block and playback ring as sxgpu_bank_read, sxgpu_iir_apply(pre), sxgpu_iir_apply(post) and
// sxgpu_bank_write(HAS_TIME, rx time + offset) -- the filter state advances on every iteration,
// also when the write is dropped as late, since the block is filtered before it is written.
//
// The decisions are bank_plan_repeat_kernel's, unchanged; this is the data kernel after it.  A
// recurrence needs whole streams per CTA, so unlike bank_repeat_data_kernel (flat vectors) a CTA
// takes kIirStreamsPerCta streams through the period in tiles of kIirTile frames (sx_iir.cuh):
//   1. coalesced: the capture (synthesised and stored to the slot, or read from an ingested
//      slot), RxCf32, into the tile's rows (a warp takes 16 vectors of two streams);
//   2. the sequential pass: lane (stream, component) runs pre cascade, hook, post cascade;
//   3. coalesced: the CF32 block stored, TxCf32, the ring stored -- by the same rules as the data
//      kernel: a block that starts on a period boundary of the ring in vectors, one that straddles
//      two slices frame by frame, nothing for a write dropped as late.
// Needs an even period and a 16-byte aligned CF32 block.  Every bank size takes this schedule.
//
// MODE: the whole iteration, or one half of it with one filter (`pre`; `post` is not used) for the
// separate calls -- sxgpu_bank_read_filtered after bank_plan_read_kernel: pass 1 as above, the
// cascade, the CF32 block stored; sxgpu_bank_write_filtered after bank_plan_write_kernel(...,
// for_data_kernel = true): the caller's CF32 block loaded, the cascade, TxCf32 and the ring by the
// rules above, and the block itself left as it was.
// ---------------------------------------------------------------------------------------
template <class Hook, int MODE = kBankModeRepeat>
__global__ void __launch_bounds__(kIirThreads) bank_repeat_iir_kernel(BankState b, char *cf32, bool capture_in_slot,
                                                                      const __grid_constant__ IirView pre,
                                                                      const __grid_constant__ IirView post, Hook hook)
{
    __shared__ __align__(16) float tile[kIirStreamsPerCta * kIirRow];
    __shared__ long long s_first[kIirStreamsPerCta], s_off[kIirStreamsPerCta], s_at[kIirStreamsPerCta];
    const uint32_t j = threadIdx.x >> 1, c = threadIdx.x & 1;
    const uint64_t s0 = uint64_t(blockIdx.x) * kIirStreamsPerCta, s = s0 + j;
    const uint32_t count = uint32_t(b.nstreams - s0 < kIirStreamsPerCta ? b.nstreams - s0 : kIirStreamsPerCta);
    const bool active = j < count;
    constexpr uint32_t kVecs = kIirTile / 2; // 16-byte vectors per row of a tile
    pdl_wait(); // the decisions, and everything before them on the stream, are in memory
    if (threadIdx.x < count) {
        if (MODE != kBankModeWrite)
            s_first[threadIdx.x] = b.rx_first_frame[s0 + threadIdx.x];
        if (MODE != kBankModeRead) {
            s_off[threadIdx.x] = b.tx_ring_offset[s0 + threadIdx.x];
            s_at[threadIdx.x] = b.tx_write_position[s0 + threadIdx.x];
        }
    }
    float zp[kIirMaxSections][2], zq[kIirMaxSections][2];
    iir_load_state(pre, s, c, active, zp);
    if (MODE == kBankModeRepeat)
        iir_load_state(post, s, c, active, zq);
    __syncthreads();

    for (uint32_t t0 = 0; t0 < b.period; t0 += kIirTile) {
        const uint32_t n = b.period - t0 < kIirTile ? b.period - t0 : kIirTile; // even
        for (uint32_t q = threadIdx.x; q < count * kVecs; q += kIirThreads) {
            const uint32_t r = q / kVecs, m = q % kVecs;
            if (2 * m >= n)
                continue;
            Pack<4> mid;
            if (MODE == kBankModeWrite) {
                mid = ld_stream<16>(cf32 + ((s0 + r) * b.period + t0 + 2 * m) * 8);
            } else {
                char *slot = b.capture_stage + ((s0 + r) * b.period + t0 + 2 * m) * 8;
                Pack<4> cap;
                if (capture_in_slot) {
                    cap = ld_stream<16>(slot);
                } else {
                    // capture_pair(b.seed + s0 + r, first) written out: through the helper the compiler
                    // associates the seed's additions differently, and read mode ran 1 % slower at 64
                    // streams (tools/bench_iir.py, B200 at a 1 000 W power limit)
                    const uint64_t first = uint64_t(s_first[r]) + t0 + 2 * m;
                    const uint64_t z0 = sx_synth_frame(b.seed + s0 + r, first), z1 = sx_synth_frame(b.seed + s0 + r, first + 1);
                    cap.w[0] = uint32_t(z0), cap.w[1] = uint32_t(z0 >> 32);
                    cap.w[2] = uint32_t(z1), cap.w[3] = uint32_t(z1 >> 32);
                    st_stream<16>(slot, cap);
                }
                RxCf32::apply<2>(cap, mid, 0.0f);
            }
            *reinterpret_cast<Pack<4> *>(&tile[r * kIirRow + 4 * m]) = mid;
        }
        __syncthreads();
        if constexpr (MODE != kBankModeRepeat) {
            IirCoeffs none; // a half runs one cascade
            none.nsections = 0;
            iir_tile_pass<2>(&tile[j * kIirRow], c, n, pre.k, zp, none, zq, NoIirHook(), s, active, t0);
        } else if constexpr (std::is_same<Hook, IdentityHook>::value) {
            iir_tile_pass<2>(&tile[j * kIirRow], c, n, pre.k, zp, post.k, zq, NoIirHook(), s, active, t0);
        } else {
            iir_tile_pass<2>(&tile[j * kIirRow], c, n, pre.k, zp, post.k, zq, hook, s, active, t0);
        }
        __syncthreads();
        for (uint32_t q = threadIdx.x; q < count * kVecs; q += kIirThreads) {
            const uint32_t r = q / kVecs, m = q % kVecs;
            if (2 * m >= n)
                continue;
            const Pack<4> mid = *reinterpret_cast<const Pack<4> *>(&tile[r * kIirRow + 4 * m]);
            const uint64_t v = t0 / 2 + m; // vector index within the block
            if (MODE != kBankModeWrite)
                st_stream<16>(cf32 + ((s0 + r) * b.period) * 8 + v * 16, mid);
            if (MODE == kBankModeRead)
                continue;
            const long long off = s_off[r];
            if (off < 0)
                continue; // discarded as late
            Pack<4> out;
            TxCf32::apply<2>(mid, out, b.thr2);
            if ((off & 1) == 0) {
                st_stream<16>(b.playback_ring + off + v * 16, out);
            } else { // straddles two slices of the time-major ring: frame by frame
                ring_store_pair(b, s0 + r, uint64_t(s_at[r]) + 2 * v, out);
            }
        }
        __syncthreads(); // the next tile overwrites the rows
    }
    iir_store_state(pre, s, c, active, zp);
    if (MODE == kBankModeRepeat)
        iir_store_state(post, s, c, active, zq);
}

// Why a filtered iteration's arguments are refused (nullptr: they are not).  A stage left out has
// nsections == 0.
inline const char *bank_repeat_iir_invalid(const BankState &b, const void *cf32, const IirView &pre, const IirView &post)
{
    if (!cf32 || reinterpret_cast<uintptr_t>(cf32) % 16)
        return "the filtered iteration needs a 16-byte aligned CF32 buffer";
    if (b.period % 2)
        return "the filtered iteration needs an even period";
    if ((pre.k.nsections && pre.nstreams != b.nstreams) || (post.k.nsections && post.nstreams != b.nstreams))
        return "a filter must have as many streams as the bank";
    if (pre.k.nsections && post.k.nsections && pre.state == post.state)
        return "the two stages cannot share one filter (and its state)";
    return nullptr;
}

// ---------------------------------------------------------------------------------------
// Launchers of the plan + data schedules.  The data kernel is launched as a programmatic
// dependent of the plan kernel, so that its launch and the first CTAs' set-up run under the
// decisions instead of after them; it waits for them with pdl_wait() before it reads them.
// ---------------------------------------------------------------------------------------
template <class... Params, class... Args>
inline cudaError_t launch_dependent(void (*kernel)(Params...), unsigned grid, unsigned block, size_t smem, cudaStream_t st,
                                    const Args &...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// The decisions of the whole iteration (MODE = kBankModeRepeat: a timed write at the read's
// timestamp + rx_time_offset_ns; `flags` and `time_ns` are not used) or of one half, one thread
// per stream, for the data kernel that follows.
template <int MODE>
inline cudaError_t launch_bank_plan(const BankState &b, char *cf32, int flags, const long long *time_ns,
                                    long long rx_time_offset_ns, cudaStream_t st)
{
    const unsigned grid = (b.nstreams + 63) / 64;
    if (MODE == kBankModeRepeat)
        bank_plan_repeat_kernel<<<grid, 64, 0, st>>>(b, cf32, rx_time_offset_ns);
    else if (MODE == kBankModeRead)
        bank_plan_read_kernel<<<grid, 64, 0, st>>>(b, cf32);
    else
        bank_plan_write_kernel<<<grid, 64, 0, st>>>(b, flags, time_ns, rx_time_offset_ns, true);
    return cudaGetLastError();
}

// The iteration or one half of it on a large bank: the decisions, then bank_repeat_data_kernel in
// that mode.  U = 16-byte vectors per thread (2 or 4).  Returns the CUDA error of the launches.
template <int MODE, int U, class Hook>
inline cudaError_t launch_bank_planned(const BankState &b, char *cf32, bool capture_in_slot, int flags, const long long *time_ns,
                                       long long rx_time_offset_ns, cudaStream_t st, const Hook &hook)
{
    const cudaError_t e = launch_bank_plan<MODE>(b, cf32, flags, time_ns, rx_time_offset_ns, st);
    if (e != cudaSuccess)
        return e;
    const uint64_t vectors = uint64_t(b.nstreams) * (b.period / 2);
    return launch_dependent(bank_repeat_data_kernel<U, Hook, MODE>, unsigned((vectors + 256 * U - 1) / (256 * U)), 256, 0, st, b,
                            cf32, capture_in_slot, hook);
}

// The iteration or one half of it with filters, every bank size: the decisions, then
// bank_repeat_iir_kernel in that mode.  A half runs `pre` alone (`post` is not used).
template <int MODE, class Hook>
inline cudaError_t launch_bank_iir(const BankState &b, char *cf32, bool capture_in_slot, int flags, const long long *time_ns,
                                   long long rx_time_offset_ns, const IirView &pre, const IirView &post, cudaStream_t st,
                                   const Hook &hook)
{
    const cudaError_t e = launch_bank_plan<MODE>(b, cf32, flags, time_ns, rx_time_offset_ns, st);
    if (e != cudaSuccess)
        return e;
    return launch_dependent(bank_repeat_iir_kernel<Hook, MODE>,
                            unsigned((uint64_t(b.nstreams) + kIirStreamsPerCta - 1) / kIirStreamsPerCta), kIirThreads, 0, st, b,
                            cf32, capture_in_slot, pre, post, hook);
}

// ---------------------------------------------------------------------------------------
// A half with a FIR filter or resampler (sxgpu_bank_read_fir, sxgpu_bank_write_fir): the same
// state, results, capture, ring, filter history and outputs as the plain half and sxgpu_fir_apply
// one after the other, without the full-rate CF32 block in memory.
//
// bank_fir_kernel<R, MODE> is fir_apply_kernel<R> (sx_fir.cuh: one warp per CTA, one tile of
// 32 R class indices of one stream per CTA, same grid, same window, same arithmetic) after the
// plan kernel, with the frames and the outputs moved:
//   read mode (after bank_plan_read_kernel): input frame i of stream s is RxCf32 of capture frame
//     i of the period -- sx_synth_frame(seed + s, rx_first_frame[s] + i), or the ingested slot --
//     and the outputs go to the caller's block as in fir_apply_kernel.  The capture slot and the
//     new history are bank_fir_read_tail_kernel's.
//   write mode (after bank_plan_write_kernel(..., for_data_kernel = true), which has written the
//     silence of forwarded-over gaps): input frames come from the caller's block, and output k,
//     through TxCf32, goes to the ring at frame tx_write_position[s] + k: at byte offset
//     tx_ring_offset[s] + 8 k when the block starts on a period boundary of the ring, frame by
//     frame through ring_frame() when it straddles two slices, nowhere when the write was dropped
//     as late.  The new history is fir_history_kernel's, from the caller's block as for apply.
//
// With an oscillator (sxgpu_bank_read_ddc, sxgpu_bank_write_duc) the full-rate frames are mixed
// (sx_nco.cuh), so that the same state, results, capture, ring, filter history, phases and outputs
// come out as from the plain half, sxgpu_nco_apply and sxgpu_fir_apply one after the other:
//   read:  input frame i of the filter is capture frame i of the period through RxCf32, mixed with
//          phi_s + i inc_s; the read tail mixes the history's new frames the same way and advances
//          phi_s.
//   write: output k of the filter is mixed with phi_s + k inc_s before TxCf32 and the ring;
//          fir_history_kernel advances phi_s, also for a stream whose write was dropped as late.
// Every read of phi_s is in the data kernel or before the tail kernel's barrier, and the phase
// advances after it.  Each kernel takes the oscillator as its template parameter Nco: NoNco for
// the plain half, NcoView with one.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float2 rx_frame(const Pack<2> &cap)
{
    Pack<2> f;
    RxCf32::apply<1>(cap, f, 0.0f);
    return make_float2(__uint_as_float(f.w[0]), __uint_as_float(f.w[1]));
}

template <int R, int MODE, class Nco>
__global__ void __launch_bounds__(32) bank_fir_kernel(BankState b, const __grid_constant__ FirCall a, bool capture_in_slot, Nco nco)
{
    extern __shared__ __align__(16) float2 win[];
    const uint64_t stream = blockIdx.x / a.chunks, chunk = blockIdx.x % a.chunks;
    pdl_wait(); // the decisions, and everything before them on the stream, are in memory
    const auto mix = nco_stream(nco, stream);
    if constexpr (MODE == kBankModeRead) {
        auto out = [&](uint64_t k, float2 v) { a.out[stream * a.nout + k] = v; };
        if (capture_in_slot) {
            const char *slot = b.capture_stage + stream * b.period * 8;
            fir_tile<R>(a, threadIdx.x, stream, chunk, win, [&](const float2 *, uint64_t i) { return mix(i, rx_frame(ld_stream<8>(slot + i * 8))); }, out);
        } else {
            const uint64_t seed = b.seed + stream, first = uint64_t(b.rx_first_frame[stream]);
            fir_tile<R>(a, threadIdx.x, stream, chunk, win, [&](const float2 *, uint64_t i) { return mix(i, rx_frame(capture_frame(seed, first + i))); }, out);
        }
    } else {
        const long long off = b.tx_ring_offset[stream];
        if (off < 0)
            return; // dropped as late: nothing is stored (the history and the phase still advance, in the tail kernel)
        const long long at = b.tx_write_position[stream];
        fir_tile<R>(a, threadIdx.x, stream, chunk, win, [](const float2 *row, uint64_t i) { return row[i]; }, [&](uint64_t k, float2 v) {
            const float2 m = mix(k, v);
            Pack<2> f, w;
            f.w[0] = __float_as_uint(m.x), f.w[1] = __float_as_uint(m.y);
            TxCf32::apply<1>(f, w, b.thr2);
            st_stream<8>((off & 1) == 0 ? b.playback_ring + off + k * 8 : ring_frame(b, stream, uint64_t(at) + k), w);
        });
    }
}

// After a read's bank_fir_kernel (or straight after the plan when the call emits nothing), one CTA
// per stream: the new history, the last hp - 1 frames of old history ++ RX(capture) (mixed as the
// data kernel mixes them), read before any of it is overwritten as in fir_history_kernel; with
// synthetic capture the whole capture slot, every frame once with the value sxgpu_bank_read stores;
// and with an oscillator the phase advanced by the period, after the barrier.  (The data kernel's
// CTAs stage overlapping windows, so none of them owns the slot's frames; here they are written in
// order.)
template <class Nco>
__global__ void __launch_bounds__(kFirHistoryThreads) bank_fir_read_tail_kernel(BankState b, const __grid_constant__ FirCall a,
                                                                                bool capture_in_slot, Nco nco)
{
    extern __shared__ __align__(16) float2 keep[]; // [hp - 1]
    const uint32_t n = a.hp - 1;
    const uint64_t s = blockIdx.x;
    char *slot = b.capture_stage + s * b.period * 8;
    const uint64_t seed = b.seed + s, first = capture_in_slot ? 0 : uint64_t(b.rx_first_frame[s]);
    float2 *hist = a.hist + s * n;
    const auto mix = nco_stream(nco, s);
    for (uint32_t i = threadIdx.x; i < n; i += kFirHistoryThreads) {
        const uint64_t k = a.nin + i; // buffer frame
        keep[i] = k < n ? hist[k] : mix(k - n, rx_frame(capture_in_slot ? ld_stream<8>(slot + (k - n) * 8) : capture_frame(seed, first + k - n)));
    }
    for (uint32_t i = threadIdx.x; i < b.period && !capture_in_slot; i += kFirHistoryThreads)
        st_stream<8>(slot + size_t(i) * 8, capture_frame(seed, first + i));
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += kFirHistoryThreads)
        hist[i] = keep[i];
    if (threadIdx.x == 0)
        nco_advance(nco, s, b.period);
}

// The data kernel of a FIR half in its R, as a programmatic dependent of the plan kernel.
template <int MODE, class Nco>
inline cudaError_t launch_bank_fir(const BankState &b, const FirCall &a, int block, size_t smem, bool capture_in_slot,
                                   const Nco &nco, cudaStream_t st)
{
    const unsigned grid = unsigned(uint64_t(b.nstreams) * a.chunks);
    if (block == 4)
        return launch_dependent(bank_fir_kernel<4, MODE, Nco>, grid, 32, smem, st, b, a, capture_in_slot, nco);
    if (block == 2)
        return launch_dependent(bank_fir_kernel<2, MODE, Nco>, grid, 32, smem, st, b, a, capture_in_slot, nco);
    return launch_dependent(bank_fir_kernel<1, MODE, Nco>, grid, 32, smem, st, b, a, capture_in_slot, nco);
}

// Lets every bank_fir_kernel with this oscillator stage a window of up to `smem` bytes.
template <class Nco>
inline cudaError_t bank_fir_allow_smem(size_t smem)
{
    for (auto kernel : {bank_fir_kernel<1, kBankModeRead, Nco>, bank_fir_kernel<2, kBankModeRead, Nco>,
                        bank_fir_kernel<4, kBankModeRead, Nco>, bank_fir_kernel<1, kBankModeWrite, Nco>,
                        bank_fir_kernel<2, kBankModeWrite, Nco>, bank_fir_kernel<4, kBankModeWrite, Nco>})
        if (const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)))
            return e;
    return cudaSuccess;
}

__global__ void bank_advance_kernel(BankState b, long long frames)
{
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < b.nstreams)
        b.clock[s] += frames;
}

} // namespace sx
