// sx_fir.cuh -- stateful FIR filters and rational resamplers for streams: real float32 taps h, an
// upsampling factor U and a downsampling factor D, applied to the I and the Q component of CF32
// samples independently, the last inputs carried from call to call.  A stream fed X frames in total
// has emitted the first ceil(X U / D) outputs of scipy.signal.upfirdn(h, x, U, D), bit for bit
// (tests/sxfir.py restates it in numpy).
//
// Polyphase form.  hp = ceil(ntaps / U) taps per phase (h zero-padded to hp U).  Output n reads the
// inputs ending at newest = (n D) div U with the taps of phase t = (n D) mod U, oldest input first:
//     acc = +0;  for j = hp-1 down to 0:  acc = acc + x[newest - j] * h[t + U j]
// every product and sum one correctly rounded float32 operation (__fmul_rn / __fadd_rn, never an
// FFMA; inputs before the stream are 0).  With g = gcd(U, D), U' = U / g and D' = D / g, output
// n = U' a + c (0 <= c < U') has newest = a D' + e_c and phase t_c, with e_c = (c D') div U' and
// t_c = g ((c D') mod U'): the outputs of one class c share their taps, and consecutive a of a class
// read inputs D' apart.
//
// A call sees its inputs behind the stream's history: buf = hist (hp - 1 frames) ++ in (nin
// frames).  The call's outputs are numbered k = c0 .. c0 + nout - 1 from the start of the current
// period of D frames (c0 = ceil(r U / D), r = frames fed so far mod D, the phase), and output k
// reads buf[k D div U - r + hp - 1 - j].  Everything the kernels need besides the buffers is a
// function of (r, nin), so a call whose nin is a multiple of D can be replayed from a graph.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "sx_nco.cuh"

namespace sx {

constexpr int kFirMaxTaps = 4096;  // SXGPU_FIR_MAX_TAPS
constexpr int kFirMaxFactor = 256; // SXGPU_FIR_MAX_FACTOR

// One call's geometry, computed on the host from the filter and (phase, nin).
struct FirCall {
    const float2 *in;   // [nstreams][nin]
    float2 *out;        // [nstreams][nout]
    float2 *hist;       // [nstreams][hp - 1], oldest first
    const float4 *taps; // [U][rows] tap table of each phase, see fir_apply_kernel
    uint64_t nin, nout;
    uint64_t c0;        // first output of the call, counted from the start of the current period
    uint64_t a_lo;      // class index a of output c0: c0 div U'
    uint64_t chunks;    // CTAs per stream
    uint32_t hp, rows;  // taps per phase; rows of a phase's tap table, (kFirBlock - 1) D' + hp
    uint32_t g, up1, down1; // gcd(U, D), U' and D'
    uint32_t phase;     // r
    uint32_t win_len;   // frames of the staged window: 32 R D' + e_max + hp
    uint32_t pad;       // 1 when R D' is even: a frame of padding after every R D' frames
};

constexpr int kFirBlock = 4; // the largest R: consecutive outputs a lane keeps in registers

// One warp per CTA.  CTA b takes chunk b mod chunks of stream b div chunks: class indices
// a = a_lo + 32 R chunk + R l + i for lane l and i < R, every class c.  The chunk's input window,
// buffer frames wb0 + o (wb0 = a_first D' - r), is staged once in shared memory in buffer order.
// Output i of lane l takes its tap s (s = hp - 1 - j, oldest input first) from window offset
// R D' l + i D' + e_c + s.  So the lane walks the offsets R D' l + e_c + q, q = 0 .. (R-1) D' + hp - 1,
// once: each input read from shared memory feeds every output i with 0 <= q - i D' < hp, with tap
// s = q - i D', and every output still meets its taps in ascending s.  The R taps of step q come in
// one 16-byte load, row q of the phase's table: taps[t][q].i = tap s = q - i D' of phase t (0 where
// that s does not exist).  In the steady part, (R-1) D' <= q < hp, every output takes a tap; at the
// two ends only the outputs whose window holds frame q add, so no product of a tap with a frame
// outside an output's own window is ever formed.  Lanes are R D' frames apart; a padding frame
// after every R D' frames makes that stride odd, so the loads of a step are conflict-free.
//
// fir_tile is that walk for one CTA, with the block's frames and the outputs' destination left to
// the kernel: in(row, i) gives input frame i < nin of the stream (row = the stream's row of a.in),
// out(k, v) stores output k of the call.
// fir_apply_kernel reads a.in and stores to a.out; the stream bank's FIR calls (sx_bank.cuh) take
// the frames from the capture and store into the playback ring.
template <int R, class In, class Out>
__device__ __forceinline__ void fir_tile(const FirCall &a, uint32_t lane, uint64_t stream, uint64_t chunk, float2 *win,
                                         const In &in, const Out &out)
{
    const uint64_t a_first = a.a_lo + chunk * (32 * R);
    const uint32_t d1 = a.down1, hp = a.hp, seg = R * d1, pad = a.pad;
    const uint64_t buf_len = a.nin + hp - 1;
    const int64_t wb0 = int64_t(a_first * d1) - int64_t(a.phase);

    // Stage buf[wb0 .. wb0 + win_len): coalesced 8-byte loads in buffer order; the first hp - 1
    // frames come from the history, frames outside the buffer are never read by a stored output
    // and are staged as zeros.
    const float2 *hist = a.hist + stream * (hp - 1);
    const float2 *row = a.in + stream * a.nin;
    for (uint32_t o = lane; o < a.win_len; o += 32) {
        const int64_t b = wb0 + int64_t(o);
        float2 v = make_float2(0.0f, 0.0f);
        if (b >= 0 && uint64_t(b) < buf_len)
            v = uint64_t(b) < hp - 1 ? hist[b] : in(row, uint64_t(b) - (hp - 1));
        win[o + (pad ? o / seg : 0)] = v;
    }
    __syncwarp();

    const uint32_t lo = (R - 1) * d1, end = lo + hp;
    for (uint32_t c = 0; c < a.up1; c++) {
        const uint32_t cd = c * d1;
        const uint32_t e = cd / a.up1, t = a.g * (cd % a.up1);
        const float4 *tab = a.taps + size_t(t) * a.rows;
        float acc_re[R], acc_im[R];
#pragma unroll
        for (int i = 0; i < R; i++)
            acc_re[i] = acc_im[i] = 0.0f;
        const float2 *p = win + lane * (seg + pad) + e + (pad ? e / seg : 0);
        uint32_t k = pad ? e % seg : 0; // offset within the current run of seg frames
        auto advance = [&]() {
            ++p;
            if (pad && ++k == seg) {
                k = 0;
                ++p;
            }
        };
        auto step = [&](uint32_t q, bool ends) {
            const float2 x = *p;
            const float4 h4 = tab[q];
            const float hs[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
            for (int i = 0; i < R; i++) {
                if (!ends || (q >= i * d1 && q - i * d1 < hp)) {
                    acc_re[i] = __fadd_rn(acc_re[i], __fmul_rn(x.x, hs[i]));
                    acc_im[i] = __fadd_rn(acc_im[i], __fmul_rn(x.y, hs[i]));
                }
            }
            advance();
        };
        uint32_t q = 0;
        for (; q < lo; q++)
            step(q, true);
        for (; q + 4 <= hp; q += 4) {
            step(q, false);
            step(q + 1, false);
            step(q + 2, false);
            step(q + 3, false);
        }
        for (; q < hp; q++)
            step(q, false);
        for (; q < end; q++)
            step(q, true);
#pragma unroll
        for (int i = 0; i < R; i++) {
            const uint64_t kk = (a_first + R * lane + i) * a.up1 + c;
            if (kk >= a.c0 && kk - a.c0 < a.nout)
                out(kk - a.c0, make_float2(acc_re[i], acc_im[i]));
        }
    }
}

template <int R>
__global__ void __launch_bounds__(32) fir_apply_kernel(const __grid_constant__ FirCall a)
{
    extern __shared__ __align__(16) float2 win[];
    const uint32_t lane = threadIdx.x;
    const uint64_t stream = blockIdx.x / a.chunks, chunk = blockIdx.x % a.chunks;
    fir_tile<R>(a, lane, stream, chunk, win, [](const float2 *row, uint64_t i) { return row[i]; },
                [&](uint64_t k, float2 v) { a.out[stream * a.nout + k] = v; });
}

// The new history, hist = buf[nin .. nin + hp - 2], after fir_apply_kernel has read the old one
// (a separate launch, so that no CTA of the apply can see a half-written history).  One CTA per
// stream: the frames that still come from the old history (nin < hp - 1) are read into shared
// memory before any is overwritten.  With an oscillator (sxgpu_bank_write_duc), thread 0 then
// advances the stream's phase by `frames`, after the barrier, as every read of it has ended.
constexpr int kFirHistoryThreads = 128;

template <class Nco = NoNco>
__global__ void __launch_bounds__(kFirHistoryThreads) fir_history_kernel(const __grid_constant__ FirCall a, Nco nco = {},
                                                                         uint32_t frames = 0)
{
    extern __shared__ __align__(16) float2 keep[]; // [hp - 1]
    const uint32_t n = a.hp - 1;
    const uint64_t stream = blockIdx.x;
    float2 *hist = a.hist + stream * n;
    const float2 *in = a.in + stream * a.nin;
    for (uint32_t i = threadIdx.x; i < n; i += kFirHistoryThreads) {
        const uint64_t b = a.nin + i; // buffer frame
        keep[i] = b < n ? hist[b] : in[b - n];
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += kFirHistoryThreads)
        hist[i] = keep[i];
    if (threadIdx.x == 0)
        nco_advance(nco, stream, frames);
}

} // namespace sx
