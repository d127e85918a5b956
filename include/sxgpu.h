/*
 * sxgpu.h -- C ABI of the B200 IQ sample-path library (libsxgpu.so).
 *
 * This is the drop-in boundary for the one data-parallel hot path of tejeez/sxxcvr's
 * SoapySX driver: the per-block conversion between S32_LE I2S frames ([I:int32][Q:int32],
 * I = left slot) and SoapySDR CF32 stream buffers ([re:f32][im:f32]).  Each entry point
 * names the reference interface it replaces (file:line under the reference tree).  The
 * binding a maintainer adds to SoapySX.cpp is shown in INTEGRATION.md.
 *
 * Conventions
 *  - plain C types only; no exceptions cross this boundary; every function returns
 *    SXGPU_OK (0) or a negative SXGPU_ERR_* code (sxgpu_strerror() names it, and
 *    sxgpu_last_error() carries the CUDA text when the code is SXGPU_ERR_CUDA);
 *  - offsets and lengths are in FRAMES (one I/Q pair), exactly as in the reference's
 *    converters; a frame is 8 bytes on the I2S side and 8 bytes as CF32 (4 as CS16);
 *  - `d_` pointers are device memory on the context's GPU, `h_` pointers host memory;
 *    the caller owns every buffer; src and dest must not overlap unless identical
 *    (in-place is allowed for the equal-width CF32 paths);
 *  - functions taking an `sxgpu_stream` are asynchronous with respect to it and may be
 *    called concurrently from several host threads as long as each thread uses its own
 *    stream; NULL selects the context's own stream, an ordinary (blocking) stream that
 *    orders with the legacy default stream like any cudaStreamCreate() stream; the *_host
 *    functions are synchronous and serialise on an internal lock;
 *  - the asynchronous functions only enqueue kernels (and, for host-resident batch
 *    descriptors, stream-ordered allocations and copies) on the given stream, so after one
 *    warm-up call they can be recorded with CUDA stream capture and replayed as a graph --
 *    the way to run a launch-bound inner loop such as one bank iteration;
 *  - there is no CPU fallback: without a usable sm_100 device sxgpu_init() fails.
 */
#ifndef SXGPU_H
#define SXGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SXGPU_ABI_VERSION 1

#define SXGPU_OK 0
#define SXGPU_ERR_INVALID (-1)     /* NULL/misaligned pointer, overflowing length, bad option */
#define SXGPU_ERR_CUDA (-2)        /* a CUDA call failed; see sxgpu_last_error() */
#define SXGPU_ERR_NO_DEVICE (-3)   /* no such GPU, or not a Blackwell sm_100 part */
#define SXGPU_ERR_NOMEM (-4)       /* device or pinned allocation failed */
#define SXGPU_ERR_UNSUPPORTED (-5) /* valid request this build does not implement */

typedef struct sxgpu_ctx sxgpu_ctx;
typedef void *sxgpu_stream; /* a cudaStream_t */

/* ---- lifetime ------------------------------------------------------------------------ */

/* One context per GPU.  Replaces nothing in the reference (which has no device state for
 * this path beyond its two staging vectors, SoapySX.cpp:552-557, :706-707); the staging
 * buffers become the context's pinned-host + device ring. */
int sxgpu_init(int device, sxgpu_ctx **out);
int sxgpu_destroy(sxgpu_ctx *ctx);
int sxgpu_abi_version(void);
const char *sxgpu_strerror(int code);
const char *sxgpu_last_error(sxgpu_ctx *ctx);

typedef struct {
    int device;
    int sm_count;
    int cc_major, cc_minor;
    uint64_t l2_bytes;
    uint64_t hbm_bytes;
    char name[64];
} sxgpu_info;
int sxgpu_device_info(sxgpu_ctx *ctx, sxgpu_info *out);

/* ---- the hot path, device-resident buffers --------------------------------------------- */

/* Replaces convert_rx_buffer(src, src_offset, dest, dest_offset, length),
 * SoapySX.cpp:103-112 (called from readStream, :957): dest[i] = 2^-31 * (float)src[i] for
 * the 2*length words of `length` frames.  Bit-exact for every input word. */
int sxgpu_convert_rx_buffer(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                            size_t dest_offset, size_t length, sxgpu_stream stream);

/* Replaces convert_tx_buffer(src, src_offset, dest, dest_offset, length, tx_threshold2),
 * SoapySX.cpp:116-137 (called from writeStream, :1090): clamp to [-1,1], scale by 2^31,
 * truncate toward zero, clear the two low bits of I and Q, then set both low bits of I
 * when fi*fi + fq*fq >= tx_threshold2 (un-fused, on the un-clamped inputs).
 * Inputs >= +1.0 and NaN, where the reference is undefined C++, follow the reference's
 * ARM deployment target: saturate to 0x7FFFFFFC, NaN -> 0 (DESIGN.md, "Parity policy"). */
int sxgpu_convert_tx_buffer(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                            size_t dest_offset, size_t length, float tx_threshold2,
                            sxgpu_stream stream);

/* EXTENSIONS -- the reference supports CF32 only (SoapySX.cpp:752-753, :1610-1616); these
 * have no reference behaviour and are specified in DESIGN.md.  CS16 frame = 2 x int16.
 * RX: out = (int16)(word >> 16).  TX: word = s << 16, flag on (s*2^-15)^2 sums. */
int sxgpu_convert_rx_buffer_cs16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset,
                                 void *d_dest, size_t dest_offset, size_t length,
                                 sxgpu_stream stream);
int sxgpu_convert_tx_buffer_cs16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset,
                                 void *d_dest, size_t dest_offset, size_t length,
                                 float tx_threshold2, sxgpu_stream stream);

/* EXTENSION -- 16-bit I2S slots: frame = [I:int16][Q:int16].  The reference only runs the
 * SX1255's 32-bit modes (its 16-bit entries are commented out as "did not work",
 * SoapySX.cpp:200-207, and ALSA is opened as S32_LE, :474), so these too have no reference
 * behaviour.  RX: f = s * 2^-15.  TX: v = trunc(2^15 * f) saturated to int16, low two bits
 * cleared, both low bits of I set when fi*fi + fq*fq >= tx_threshold2. */
int sxgpu_convert_rx_buffer_s16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                                size_t dest_offset, size_t length, sxgpu_stream stream);
int sxgpu_convert_tx_buffer_s16(sxgpu_ctx *ctx, const void *d_src, size_t src_offset, void *d_dest,
                                size_t dest_offset, size_t length, float tx_threshold2,
                                sxgpu_stream stream);

/* Many independent blocks in one launch: what a bank of SoapySX devices would do as one
 * convert_*_buffer call each per period (256 frames by default, SoapySX.cpp:451).
 * `blocks` is read on the host when blocks_on_device == 0 (it is then copied into the
 * stream-ordered staging memory), or is a device pointer when blocks_on_device != 0.
 * max_length = longest block in frames; it picks the work split (a warp per block up to
 * 4096 frames, slices of CTAs per block above) and may be 0 for host-resident lists. */
typedef struct {
    const void *src;      /* device pointer, first frame of the block */
    void *dest;           /* device pointer, first frame of the block */
    uint64_t length;      /* frames */
    float tx_threshold2;  /* TX only */
    uint32_t reserved;
} sxgpu_block;
int sxgpu_convert_rx_batch(sxgpu_ctx *ctx, const sxgpu_block *blocks, uint32_t nblocks,
                           int blocks_on_device, size_t max_length, sxgpu_stream stream);
int sxgpu_convert_tx_batch(sxgpu_ctx *ctx, const sxgpu_block *blocks, uint32_t nblocks,
                           int blocks_on_device, size_t max_length, sxgpu_stream stream);

/* Repeater path (example/linear_repeater.py:50-71 with an identity process()): RX-convert
 * `length` frames and TX-convert the result in one pass.  The CF32 intermediate is an
 * API-visible buffer in the reference, so it is written to d_cf32 unless that is NULL. */
int sxgpu_convert_loopback(sxgpu_ctx *ctx, const void *d_i2s_in, void *d_cf32, void *d_i2s_out,
                           size_t length, float tx_threshold2, sxgpu_stream stream);

/* Silence for the gaps between timed TX bursts: what ALSA plays for regions that were
 * forwarded over (silence_size = boundary, SoapySX.cpp:493-496) -- all-zero I2S words. */
int sxgpu_fill_silence(sxgpu_ctx *ctx, void *d_i2s, size_t offset, size_t length,
                       sxgpu_stream stream);

/* ---- a bank of streams resident in HBM ---------------------------------------------------- */

/* Thousands of independent RX/TX stream pairs served per launch.  Each stream of the bank
 * behaves like one activated SoapySX device in its default stream mode: sxgpu_bank_read is
 * readStream(rx, buf, period) and sxgpu_bank_write is writeStream(tx, buf, period, flags,
 * timeNs) (SoapySX.cpp:868-1105) applied to every stream at once, with the same overrun
 * skip, timestamping, late-burst discard, underrun forward and silence rules -- but the
 * frame counters, the playback ring and the sample buffers all stay in device memory and the
 * bookkeeping runs as a kernel (one thread per stream).  The I2S hardware is the same
 * deterministic stand-in as on the host: stream s captures sx_synth_frame(seed + s, k), and
 * its sample clock moves when a blocking transfer must wait or when sxgpu_bank_advance says so. */
typedef struct sxgpu_bank sxgpu_bank;
typedef struct {
    uint32_t nstreams;
    uint32_t period;       /* frames per block; 0 = 256, capped at 65536 (SoapySX.cpp:451, :464-466) */
    double sample_rate;    /* Hz; feeds every timestamp */
    float tx_threshold2;
    uint32_t reserved;
    uint64_t seed;
} sxgpu_bank_config;
int sxgpu_bank_create(sxgpu_ctx *ctx, const sxgpu_bank_config *config, sxgpu_bank **out);
int sxgpu_bank_destroy(sxgpu_bank *bank); /* before sxgpu_destroy of its context, which refuses otherwise */
/* Let `frames` sample periods pass on every stream. */
int sxgpu_bank_advance(sxgpu_bank *bank, int64_t frames, sxgpu_stream stream);
/* d_cf32: [nstreams][period] CF32 samples on the device. */
int sxgpu_bank_read(sxgpu_bank *bank, void *d_cf32, sxgpu_stream stream);
/* flags: SOAPY_SDR_HAS_TIME (4) or 0.  With HAS_TIME, stream s is written at d_time_ns[s], or,
 * when d_time_ns is NULL, at the timestamp its last read returned plus rx_time_offset_ns. */
int sxgpu_bank_write(sxgpu_bank *bank, const void *d_cf32, int flags, const long long *d_time_ns,
                     long long rx_time_offset_ns, sxgpu_stream stream);
/* The repeater iteration without its filters (example/linear_repeater.py:50-71 with an identity
 * process()) in one launch: sxgpu_bank_read(bank, d_cf32) followed by sxgpu_bank_write(bank,
 * d_cf32, SOAPY_SDR_HAS_TIME, NULL, rx_time_offset_ns).  Same state, results, CF32 block and
 * playback ring as the two calls; each stream's three stages run back to back on one warp, so the
 * intermediate reads are served from L2 and only the writes reach HBM.  With the script's channel
 * filters: sxgpu_bank_repeat_filtered below. */
int sxgpu_bank_repeat(sxgpu_bank *bank, void *d_cf32, long long rx_time_offset_ns, sxgpu_stream stream);
/* The same iteration split around DSP of the caller's own (the process(buf) of
 * example/linear_repeater.py:62): begin = sxgpu_bank_read with the CF32 block marked persisting
 * in L2 for `stream`; the caller then launches its kernel(s) on that stream, in place on d_cf32;
 * end = sxgpu_bank_write(bank, d_cf32, SOAPY_SDR_HAS_TIME, NULL, rx_time_offset_ns) and the mark
 * is lifted.  DSP that is memoryless per sample can instead be compiled INTO the one-launch
 * iteration, between the two filters of sxgpu_bank_repeat_filtered: include/sx_hook.cuh. */
int sxgpu_bank_repeat_begin(sxgpu_bank *bank, void *d_cf32, sxgpu_stream stream);
int sxgpu_bank_repeat_end(sxgpu_bank *bank, const void *d_cf32, long long rx_time_offset_ns, sxgpu_stream stream);
/* Frames from outside instead of the synthetic capture: copy one period of I2S frames for each
 * of `nstreams` consecutive streams, i2s[stream - first_stream][period], into their capture
 * slots.  `i2s` may be pinned or pageable host memory or device memory; the copy is ordered on
 * `stream`.  From the first call on (nstreams == 0 just switches the mode) the bank no longer
 * synthesises: sxgpu_bank_read / sxgpu_bank_repeat convert whatever the slots hold, with the
 * same bookkeeping.  This is the entry for frames produced by real front-ends (or by N host-side
 * ALSA stand-ins): what snd_pcm_readi delivers in SoapySX.cpp:948, for many streams at once. */
int sxgpu_bank_ingest(sxgpu_bank *bank, uint32_t first_stream, uint32_t nstreams, const void *i2s,
                      sxgpu_stream stream);
/* The other end: for each of `nstreams` consecutive streams copy the last `nframes` frames it
 * wrote (the frames ending at its TX counter; silence before frame 0) out of its playback ring
 * to i2s[stream - first_stream][nframes] -- what snd_pcm_writei would be handed in
 * SoapySX.cpp:1093.  `i2s`: device memory, or pinned host memory (written across PCIe by the
 * kernel itself).  Asynchronous on `stream`. */
int sxgpu_bank_drain(sxgpu_bank *bank, uint32_t first_stream, uint32_t nstreams, size_t nframes, void *i2s,
                     sxgpu_stream stream);
/* For include/sx_hook.cuh: the bank's device-side view (struct sx::BankState), so that a fused
 * iteration with a user functor compiled into it can be launched from the caller's own
 * translation unit.  out_bytes must be sizeof(sx::BankState). */
int sxgpu_bank_device_view(sxgpu_bank *bank, void *out, size_t out_bytes, int *external_capture);
/* Per-stream results of the last read / write and the counters, copied to host arrays of
 * nstreams elements (any pointer may be NULL).  These synchronise with `stream`. */
int sxgpu_bank_last_read(sxgpu_bank *bank, int32_t *h_ret, int32_t *h_flags, int64_t *h_time_ns,
                         sxgpu_stream stream);
int sxgpu_bank_last_write(sxgpu_bank *bank, int32_t *h_ret, sxgpu_stream stream);
int sxgpu_bank_positions(sxgpu_bank *bank, int64_t *h_clock, int64_t *h_rx_position,
                         int64_t *h_tx_position, sxgpu_stream stream);
/* Copy `nframes` I2S frames of stream `index`'s playback ring, starting at frame counter
 * `position`, to the host.  Only the most recent ring_frames positions are still held. */
int sxgpu_bank_playback(sxgpu_bank *bank, uint32_t index, int64_t position, size_t nframes,
                        void *h_i2s, sxgpu_stream stream);
int sxgpu_bank_ring_frames(sxgpu_bank *bank, uint64_t *ring_frames);

/* ---- stateful IIR filters for a bank's streams ------------------------------------------- */

/* The channel filters of the reference repeater (example/linear_repeater.py:78-109): a cascade of
 * second-order sections with real coefficients, applied to I and Q independently, the state
 * carried from block to block -- scipy.signal.sosfilt(sos, x, zi=state) with a real `sos` on
 * complex x, one filter state per stream.  Float32 arithmetic in scipy's transposed direct form II,
 * operation for operation (DESIGN.md, "Parity policy"): the same bits as sosfilt on complex64
 * input with the float32-rounded coefficients. */
#define SXGPU_IIR_MAX_SECTIONS 8
typedef struct sxgpu_iir sxgpu_iir; /* per-stream cascade state in device memory, one per bank stream */
/* sos: nsections rows of scipy's layout, b0 b1 b2 a0 a1 a2, as double; rounded to float32 once,
 * here.  a0 must be exactly 1 and every coefficient finite; 1 <= nsections <= 8 (order 16).
 * The state starts at zero.  sxgpu_destroy of the context refuses while a filter is alive. */
int sxgpu_iir_create(sxgpu_ctx *ctx, uint32_t nstreams, uint32_t nsections, const double *sos, sxgpu_iir **out);
int sxgpu_iir_destroy(sxgpu_iir *f);
/* zi / zf: scipy's layout for x of shape (nstreams, n) filtered along the last axis, that is
 * [nsections][nstreams][2] complex64 on the host.  NULL zi = zeros.  Both synchronise with `stream`. */
int sxgpu_iir_set_state(sxgpu_iir *f, const void *h_zi, sxgpu_stream stream);
int sxgpu_iir_get_state(sxgpu_iir *f, void *h_zf, sxgpu_stream stream);
/* Filter d_cf32[nstreams][period] in place, carrying the state: sosfilt(sos, x, zi=state) per
 * stream.  1 <= period <= 65536; d_cf32 8-byte aligned device memory. */
int sxgpu_iir_apply(sxgpu_iir *f, void *d_cf32, uint32_t period, sxgpu_stream stream);
/* The repeater iteration with its filters: read -> pre -> post -> CF32 block and timed write.
 * Same state, results, positions, CF32 block and playback ring, bit for bit, as sxgpu_bank_read,
 * sxgpu_iir_apply(pre), sxgpu_iir_apply(post), sxgpu_bank_write(bank, d_cf32, SOAPY_SDR_HAS_TIME,
 * NULL, rx_time_offset_ns); both filters advance on every iteration, also when the write is
 * dropped as late.  Either filter may be NULL (both NULL: exactly sxgpu_bank_repeat).  Needs filters
 * of the bank's stream count, two different filters, an even period and a 16-byte aligned d_cf32. */
int sxgpu_bank_repeat_filtered(sxgpu_bank *bank, sxgpu_iir *pre, sxgpu_iir *post, void *d_cf32,
                               long long rx_time_offset_ns, sxgpu_stream stream);
/* The two halves with a filter fused in, for a bank used only as receivers or only as transmitters,
 * and for the repeater split around DSP of the caller's own: read_filtered(pre), the caller's
 * kernels on d_cf32, then write_filtered(post, SOAPY_SDR_HAS_TIME, NULL, rx_time_offset_ns) is the
 * filtered repeater iteration with that DSP between its filters.  Each is one pass over the CF32
 * block instead of two.  Same requirements as sxgpu_bank_repeat_filtered: a filter of this context
 * with the bank's stream count, an even period and a 16-byte aligned d_cf32 (checked also when f is
 * NULL).
 * sxgpu_bank_read, then sxgpu_iir_apply(f, d_cf32, period): the same state, results, positions,
 * capture and CF32 block, bit for bit, in one pass.  f NULL: exactly sxgpu_bank_read. */
int sxgpu_bank_read_filtered(sxgpu_bank *bank, sxgpu_iir *f, void *d_cf32, sxgpu_stream stream);
/* The caller's block filtered by f and then written as sxgpu_bank_write(bank, ., flags, d_time_ns,
 * rx_time_offset_ns) would write it.  d_cf32 is not modified.  f's state advances also when a
 * stream's write is dropped as late.  f NULL: exactly sxgpu_bank_write. */
int sxgpu_bank_write_filtered(sxgpu_bank *bank, sxgpu_iir *f, const void *d_cf32, int flags,
                              const long long *d_time_ns, long long rx_time_offset_ns, sxgpu_stream stream);
/* For include/sx_hook.cuh, like sxgpu_bank_device_view: the filter's device-side view (struct
 * sx::IirView).  out_bytes must be sizeof(sx::IirView). */
int sxgpu_iir_device_view(sxgpu_iir *f, void *out, size_t out_bytes);

/* ---- the hot path, host buffers ---------------------------------------------------------- */

/* Same contracts as the two converters above, but src and dest are HOST memory, as they
 * are at the reference's call sites (buffer_rx/buffs[0], SoapySX.cpp:957, :1090).  The
 * host->device copy, the kernel and the device->host copy all happen inside the call,
 * pipelined in chunks over the context's ring.  Pinned (cudaHostAlloc / registered)
 * buffers are used in place; pageable buffers are bounced through pinned staging; up to
 * 2^18 frames of pinned memory are converted by one kernel that reads and writes the host
 * buffers across PCIe itself.  Either side may also be DEVICE memory of the context's GPU
 * (a torch / cupy buffer handed to readStream or writeStream): that side's copy is skipped
 * and the kernel uses the buffer directly. */
int sxgpu_convert_rx_buffer_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                 void *h_dest, size_t dest_offset, size_t length);
/* The same while the source is still being filled (a readStream of many ALSA rings' worth of frames:
 * snd_pcm_readi copies piece by piece, SoapySX.cpp:948, and the conversion of the first pieces need
 * not wait for the last).  *frames_ready = frames of the block in place so far, written by the
 * filling thread with release semantics; bit 63 set = that count is final, the block ends there.
 * No chunk of the pipeline is touched before its frames are in place.  Returns when everything
 * that came is converted; *converted (may be NULL) = how many frames that was. */
int sxgpu_convert_rx_buffer_host_gated(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                       size_t dest_offset, size_t length, const volatile uint64_t *frames_ready,
                                       size_t *converted);
int sxgpu_convert_tx_buffer_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                 void *h_dest, size_t dest_offset, size_t length,
                                 float tx_threshold2);

/* EXTENSION (no reference behaviour): the CS16 conversions with host buffers. */
int sxgpu_convert_rx_buffer_cs16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                      void *h_dest, size_t dest_offset, size_t length);
int sxgpu_convert_tx_buffer_cs16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset,
                                      void *h_dest, size_t dest_offset, size_t length,
                                      float tx_threshold2);

/* EXTENSION (no reference behaviour): the 16-bit I2S slot conversions with host buffers. */
int sxgpu_convert_rx_buffer_s16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                     size_t dest_offset, size_t length);
int sxgpu_convert_tx_buffer_s16_host(sxgpu_ctx *ctx, const void *h_src, size_t src_offset, void *h_dest,
                                     size_t dest_offset, size_t length, float tx_threshold2);

/* ---- statistics (off the hot path) ------------------------------------------------------- */

/* Order-sensitive checksum and flag counts over 32-bit words; every field is a sum mod 2^64
 * (or an xor), so shards reduce in any order.  Used for full-size parity checks and for the
 * cross-GPU gather.  Synchronous: returns with *h_out filled. */
typedef struct {
    uint64_t sum;    /* sum of words */
    uint64_t wsum;   /* sum of word * (2*(base_index+i)+1) */
    uint64_t x;      /* xor of words */
    uint64_t count;  /* words */
    uint64_t tx_on;  /* even-index words with bit 1 set: TX-enable flag, SoapySX.cpp:126-133 */
    uint64_t rail;   /* words whose upper 30 bits are 0x7FFFFFFC or 0x80000000 */
} sxgpu_stats;
int sxgpu_stats_words(sxgpu_ctx *ctx, const void *d_words, size_t nwords, uint64_t base_index,
                      sxgpu_stats *h_out, sxgpu_stream stream);

/* ---- synthetic capture source (stands in for the SX1255 ADC) ------------------------------ */

/* Frame k = sx_synth_frame(seed, k): identical to what the host-side ALSA stub produces. */
int sxgpu_synth_frames(sxgpu_ctx *ctx, void *d_i2s, uint64_t first_frame, size_t nframes,
                       uint64_t seed, sxgpu_stream stream);

/* ---- memory and stream plumbing for C/C++ hosts ------------------------------------------- */

int sxgpu_malloc(sxgpu_ctx *ctx, void **d_ptr, size_t bytes);
int sxgpu_free(sxgpu_ctx *ctx, void *d_ptr);
int sxgpu_malloc_host(sxgpu_ctx *ctx, void **h_ptr, size_t bytes); /* pinned, on the GPU's NUMA node */
int sxgpu_free_host(sxgpu_ctx *ctx, void *h_ptr);
int sxgpu_host_register(sxgpu_ctx *ctx, void *h_ptr, size_t bytes); /* pin caller memory */
int sxgpu_host_unregister(sxgpu_ctx *ctx, void *h_ptr);
int sxgpu_memcpy_h2d(sxgpu_ctx *ctx, void *d_dst, const void *h_src, size_t bytes,
                     sxgpu_stream stream);
int sxgpu_memcpy_d2h(sxgpu_ctx *ctx, void *h_dst, const void *d_src, size_t bytes,
                     sxgpu_stream stream);
int sxgpu_stream_create(sxgpu_ctx *ctx, sxgpu_stream *out);
int sxgpu_stream_destroy(sxgpu_ctx *ctx, sxgpu_stream stream);
int sxgpu_stream_sync(sxgpu_ctx *ctx, sxgpu_stream stream); /* NULL = context stream */

/* ---- several GPUs from one process ----------------------------------------------------------- */

/* One context and one host thread per GPU of `devices` (each ordinal once).  The path shards
 * trivially -- every output word depends on one input word or one I/Q pair (SoapySX.cpp:108-111,
 * :121-136), streams have independent counters (:378) -- so nothing crosses between GPUs and
 * there is no collective: a list of blocks is split, every GPU converts its share at once.
 * One multi-GPU call at a time per object; the per-GPU contexts (sxgpu_multi_context) stay usable
 * on their own, e.g. for sxgpu_stats_words on each GPU's output. */
typedef struct sxgpu_multi sxgpu_multi;
int sxgpu_multi_create(const int *devices, int ndevices, sxgpu_multi **out);
int sxgpu_multi_destroy(sxgpu_multi *m);
int sxgpu_multi_size(sxgpu_multi *m);
sxgpu_ctx *sxgpu_multi_context(sxgpu_multi *m, int index);
const char *sxgpu_multi_last_error(sxgpu_multi *m);
/* HOST buffers (src / dest of every block are host pointers; tx_threshold2 per block): block b is
 * converted by GPU b mod G through that GPU's host pipeline, all GPUs in parallel, each driven by
 * its own thread.  Synchronous: returns when every block is done. */
int sxgpu_multi_convert_rx_host(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks);
int sxgpu_multi_convert_tx_host(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks);
/* DEVICE buffers: every block is converted on the GPU its source buffer lives on (its destination
 * must be on the same GPU), one batched launch per GPU on that GPU's context stream.
 * Asynchronous; sxgpu_multi_sync waits for every GPU. */
int sxgpu_multi_convert_rx_batch(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks);
int sxgpu_multi_convert_tx_batch(sxgpu_multi *m, const sxgpu_block *blocks, uint32_t nblocks);
int sxgpu_multi_sync(sxgpu_multi *m);

/* ---- tuning and accounting ---------------------------------------------------------------- */

/* Options (all have measured defaults; see DESIGN.md):
 *   "rx_variant", "tx_variant"  0 = auto (= 4), 1 = 128-bit vector, 2 = 256-bit vector,
 *                               3 = bulk-async (TMA) staged through shared memory -- those three
 *                               on persistent grids -- 4 = vector accesses, one tile per CTA,
 *                               CTAs handed out in order by the hardware
 *   "ctas_per_sm"               persistent grid = sm_count * ctas_per_sm (0 = auto)
 *   "host_chunk_frames"         chunk size of the *_host pipeline
 *   "host_mode"                 0 = auto, 1 = copy-engine pipeline, 2 = zero-copy kernel
 *   "resident_max_frames"       0 = off (default).  N > 0: synchronous CF32 calls of up to N
 *                               frames on host buffers are served by a resident single-CTA
 *                               kernel through a doorbell in pinned memory instead of a kernel
 *                               launch each (period-sized blocks, SoapySX.cpp:451); the kernel
 *                               leaves after 2 ms without work, after 20 ms in any case, and at
 *                               once when the library is about to synchronise the device
 *   "bank_repeat_variant"       schedule of sxgpu_bank_repeat: 0 = auto (by stream count),
 *                               K in {1, 2, 4, 8} = a warp takes K streams per round, stage by
 *                               stage through memory; 100 = a CTA takes 32 streams per round;
 *                               200 + K, K in {1, 2, 4} = a warp takes K streams per round and
 *                               keeps every intermediate in registers (stores only); 300, 302,
 *                               303 = the same with a CTA's first warp deciding for 32 streams;
 *                               600, 604 = decisions by a thread-per-stream kernel, then
 *                               the samples by CTAs that take one chunk each (2 or 4 vectors per
 *                               thread), the second kernel a programmatic dependent of the first
 *                               ("bank_pdl" = 0 turns that off)
 *   "batch_variant"             blocks above 4096 frames in sxgpu_convert_*_batch: 0 = auto
 *                               (2 when the blocks are of similar length, else 3), 1 = slices of
 *                               CTAs on vector accesses, 2 = one chunk per CTA in block-then-chunk
 *                               order, 3 = tiles of all blocks on the bulk-async schedule
 *   "loopback_variant"          sxgpu_convert_loopback: 0 = auto (= 2), 1 = vector accesses on a
 *                               persistent grid, 2 = vector accesses, one tile per CTA,
 *                               3 = bulk-async
 *   "small_mode"                completion of synchronous calls of up to zero_copy_max_frames
 *                               frames on host buffers: 0 = auto (= 2), 1 = stream
 *                               synchronisation, 2 = the kernel raises a flag in pinned memory
 *                               that the caller spins on
 *   "host_chunk_min_frames"     first and last chunk of the *_host pipeline; chunk sizes double
 *                               from here up to host_chunk_frames and mirror at the end
 *                               (0 = uniform chunks)
 *   "bounce_threads"            threads that share the copy of a pageable caller buffer to or
 *                               from pinned staging in the *_host calls (copies of 2 MiB and more):
 *                               0 = auto (half of the hardware threads, shared between the
 *                               LOCAL_WORLD_SIZE ranks of a torchrun job, at most 8),
 *                               1 = the calling thread alone
 *   "numa_local_alloc"          1 (default): pinned host memory this library allocates
 *                               (sxgpu_malloc_host, the bounce buffers of the *_host pipeline) is
 *                               faulted in while the calling thread is confined to the CPUs next to
 *                               the GPU, so it lands on the GPU's NUMA node; the thread's affinity
 *                               is restored before the call returns.  0 = leave placement alone
 *   "numa_node"                 read-only: the GPU's NUMA node, -1 if the system reports none
 */
int sxgpu_set_option(sxgpu_ctx *ctx, const char *key, int64_t value);
int sxgpu_get_option(sxgpu_ctx *ctx, const char *key, int64_t *value);
/* Counters: "launches" (kernels launched by this context), "frames_rx", "frames_tx",
 * "h2d_bytes", "d2h_bytes", "resident_launches", "resident_calls", "flagged_calls". */
int sxgpu_get_counter(sxgpu_ctx *ctx, const char *key, uint64_t *value);

#ifdef __cplusplus
}
#endif
#endif /* SXGPU_H */
