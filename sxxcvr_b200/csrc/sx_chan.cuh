// sx_chan.cuh -- polyphase DFT channelizers for streams: every stream split into M channel-rate
// streams, channel k centred at k / M cycles per input sample (k >= M/2: (k - M) / M, numpy's fft
// order), decimated by D (D divides M), with one real prototype low-pass h of ntaps taps and the
// last ntaps - 1 inputs carried from call to call (tests/sxchan.py restates it in numpy).  A stream
// fed X frames in total has emitted outputs m = 0 .. ceil(X / D) - 1 of every channel,
//     y_k[m] = sum_j h[j] x[m D - j] e^{-j 2 pi k (m D - j) / M}      (x before frame 0 is 0)
// computed in float32, bit for bit, as follows (N = m D; every product and sum one correctly
// rounded operation, __fmul_rn / __fadd_rn / __fsub_rn, never an FFMA; I and Q separately):
//   1. branch sums, r = 0 .. M-1, P_r = ceil((ntaps - r) / M) taps (0 when r >= ntaps):
//          u_r = +0;  for p = P_r - 1 down to 0:  u_r = u_r + x[N - p M - r] * h[p M + r]
//   2. a[i] = u_{(N - rev(i)) mod M}, rev reversing the log2 M bits of i;
//   3. radix-2 decimation in time, stages h = 1, 2, .. M/2: for every i with (i mod 2h) < h,
//          w = T[(i mod 2h) M / (2h)],  t = a[i+h] w,  a[i] = a[i] + t,  a[i+h] = a[i] - t
//      with t.re = q.re w.re - q.im w.im and t.im = q.re w.im + q.im w.re (q = a[i+h]), also for
//      w = T[0]; T[j] is the oscillator's coarse table conjugated, (A[q].re, -A[q].im), q = j 1024 / M;
//   4. y_k[m] = a[k].
//
// A call sees its inputs behind the history: buf = hist (ntaps - 1 frames) ++ in (nin frames).
// With r = X mod M before the call (the phase), the call's outputs are numbered o = 0 .. nout - 1;
// output o has its newest frame at call frame e0 + o D, buffer frame e0 + o D + ntaps - 1, with
// e0 = (D - r mod D) mod D, and N mod M = (r + e0 + o D) mod M.  Everything the kernel needs
// besides the buffers is a function of (r, nin), so a call whose nin is a multiple of M can be
// replayed from a graph.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace sx {

constexpr int kChanMaxChannels = 1024; // SXGPU_CHAN_MAX_CHANNELS: the coarse table's resolution
constexpr int kChanMaxTaps = 16384;    // SXGPU_CHAN_MAX_TAPS
constexpr int kChanBlock = 4;          // outputs of one branch a thread keeps in registers

// One call's geometry, computed on the host from the channelizer and (phase, nin).
struct ChanCall {
    const float2 *in;   // [nstreams][nin]
    float2 *out;        // [nstreams][M][nout]
    const float2 *hist; // [nstreams][ntaps - 1], oldest first
    const float *taps;  // [ntaps], float32
    const float2 *tw;   // [1024]: the coarse table conjugated, so T[j] is tw[j 1024 / M]
    uint64_t nin, nout;
    uint64_t tiles;     // CTAs per stream
    uint32_t m, log2m, down, ntaps;
    uint32_t groups;    // G: a CTA has M G threads and takes T = kChanBlock G consecutive outputs
    uint32_t win_len;   // frames of the staged window, (T - 1) D + ntaps
    uint32_t e0;        // call frames before the newest frame of output 0
    uint32_t rot0;      // N mod M of output 0
};

// CTA b takes tile b mod tiles of stream b div tiles: outputs o = T tile + t, t < T.  Its input
// window, buffer frames T tile D + e0 + w, w < win_len, is staged once in shared memory with
// coalesced 8-byte loads (the first ntaps - 1 buffer frames from the history; frames past the
// buffer feed only outputs that are not stored, and are staged as zeros).  Thread (g, r), r = its
// index mod M, sums branch r of outputs t = g + j G, j < kChanBlock: window frame
// t D + ntaps - 1 - p M - r with tap h[p M + r], the tap loaded once for the four outputs.  The
// lanes of a warp take consecutive r, so their frames are consecutive: no bank conflicts.  Once
// every sum is formed the window is dead; the sums are written over it, output t's a[] in row t
// (M + 1 frames apart, so that the stores, which walk a channel's outputs, are conflict-free), each
// u_r to slot rev((N - r) mod M).  The log2 M stages then run in place in shared memory, a barrier
// after each, and the tile is stored channel-major: for each channel the T outputs are contiguous.
__global__ void __launch_bounds__(1024) chan_apply_kernel(const __grid_constant__ ChanCall a)
{
    extern __shared__ __align__(16) float2 sm[];
    const uint32_t tid = threadIdx.x, nthreads = blockDim.x;
    const uint64_t stream = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;
    const uint32_t M = a.m, G = a.groups, T = kChanBlock * G, hn = a.ntaps - 1;

    const uint64_t wb0 = tile * T * a.down + a.e0, buf_len = a.nin + hn;
    const float2 *hist = a.hist + stream * hn;
    const float2 *row = a.in + stream * a.nin;
    for (uint32_t w = tid; w < a.win_len; w += nthreads) {
        const uint64_t b = wb0 + w;
        float2 v = make_float2(0.0f, 0.0f);
        if (b < buf_len)
            v = b < hn ? hist[b] : row[b - hn];
        sm[w] = v;
    }
    __syncthreads();

    const uint32_t r = tid & (M - 1), g = tid >> a.log2m;
    const uint32_t np = r < a.ntaps ? (a.ntaps - r + M - 1) >> a.log2m : 0;
    float acc_re[kChanBlock], acc_im[kChanBlock];
#pragma unroll
    for (int j = 0; j < kChanBlock; j++)
        acc_re[j] = acc_im[j] = 0.0f;
    const float2 *x = sm + g * a.down + hn - r;
    const float *h = a.taps + r;
    for (uint32_t p = np; p-- > 0;) {
        const float hv = __ldg(h + p * M);
        const float2 *xp = x - p * M;
#pragma unroll
        for (int j = 0; j < kChanBlock; j++) {
            const float2 v = xp[j * G * a.down];
            acc_re[j] = __fadd_rn(acc_re[j], __fmul_rn(v.x, hv));
            acc_im[j] = __fadd_rn(acc_im[j], __fmul_rn(v.y, hv));
        }
    }
    __syncthreads();

    const uint32_t stride = M + 1;
#pragma unroll
    for (int j = 0; j < kChanBlock; j++) {
        const uint32_t t = g + j * G;
        const uint32_t nmod = uint32_t((a.rot0 + ((tile * T + t) & (M - 1)) * a.down) & (M - 1));
        const uint32_t slot = __brev((nmod - r) & (M - 1)) >> (32 - a.log2m);
        sm[t * stride + slot] = make_float2(acc_re[j], acc_im[j]);
    }
    __syncthreads();

    const uint32_t half = M >> 1, nbf = T * half;
    for (uint32_t s = 0; s < a.log2m; s++) {
        const uint32_t hs = 1u << s;
        for (uint32_t b = tid; b < nbf; b += nthreads) {
            const uint32_t t = b >> (a.log2m - 1), bb = b & (half - 1), jj = bb & (hs - 1);
            float2 *pa = sm + t * stride + ((bb >> s) << (s + 1)) + jj;
            const float2 w = __ldg(a.tw + (jj << (9 - s)));
            const float2 p = pa[0], q = pa[hs];
            const float tr = __fsub_rn(__fmul_rn(q.x, w.x), __fmul_rn(q.y, w.y));
            const float ti = __fadd_rn(__fmul_rn(q.x, w.y), __fmul_rn(q.y, w.x));
            pa[0] = make_float2(__fadd_rn(p.x, tr), __fadd_rn(p.y, ti));
            pa[hs] = make_float2(__fsub_rn(p.x, tr), __fsub_rn(p.y, ti));
        }
        __syncthreads();
    }

    const uint32_t log2t = __ffs(T) - 1;
    for (uint32_t e = tid; e < T * M; e += nthreads) {
        const uint32_t k = e >> log2t, t = e & (T - 1);
        const uint64_t o = tile * T + t;
        if (o < a.nout)
            a.out[(stream * M + k) * a.nout + o] = sm[t * stride + k];
    }
}

// ---- the synthesis (transmit) channelizer: M channel-rate streams combined into one ----------
// The adjoint of the above (tests/sxchansynth.py restates it).  With D = up dividing M, hp =
// ceil(ntaps / D) and X the input frames per channel fed before, output frame n = m D + t (t < D)
// of a stream is
//     x[n] = sum_k sum_m h[n - m D] y_k[m] e^{+j 2 pi k n / M}            (y before frame 0 is 0)
// computed in float32, bit for bit, as follows (the same roundings as chan_apply_kernel):
//   1. for every input frame m, Y_m = the unnormalised M-point inverse DFT of (y_0[m] .. y_{M-1}[m]):
//      a[i] = y_{rev(i)}[m], then the radix-2 decimation-in-time stages of chan_apply_kernel with
//      T+[j] = A[j 1024 / M], the oscillator's coarse table not conjugated, and Y_m[i] = a[i];
//   2. P_t = ceil((ntaps - t) / D) (0 when t >= ntaps):
//          acc = +0;  for p = P_t - 1 down to 0:  acc = acc + Y_{m-p}[n mod M] * h[t + p D]
//
// A call sees each channel's inputs behind its history: buf = hist (hp - 1 frames) ++ in (nin
// frames).  With r = X mod (M / D) before the call (the phase), output o = j D + t of the call reads
// buffer frames j + hp - 1 - p, and n mod M = (r D + o) mod M.  Everything the kernel needs besides
// the buffers is a function of (r, nin), so a call whose nin is a multiple of M / D can be replayed
// from a graph.
constexpr int kChanSynthBlock = 8; // outputs a thread keeps in registers

// One call's geometry, computed on the host from the synthesizer and (phase, nin).
struct ChanSynthCall {
    const float2 *in;   // [nstreams][M][nin]
    float2 *out;        // [nstreams][nin D]
    const float2 *hist; // [nstreams][M][hp - 1], raw inputs, oldest first
    const float *taps;  // [ntaps], float32
    const float2 *tw;   // [1024]: the coarse table, so T+[j] is tw[j 1024 / M]
    uint64_t nin;
    uint64_t tiles;     // CTAs per stream
    uint32_t m, log2m, log2up, ntaps, hp;
    uint32_t frames;    // B: input frames of a tile, so B D outputs
    uint32_t chunk;     // F: window frames staged and transformed at once
    uint32_t rot0;      // r D mod M: n mod M of output 0
};

// CTA b takes tile b mod tiles of stream b div tiles: the call's input frames B tile + j, j < B, and
// outputs o = B D tile + l, l < B D.  Thread tid keeps outputs l = tid + i blockDim.x, i <
// kChanSynthBlock.  The tile's window is its own frames behind the hp - 1 before them (window frame
// w = buffer frame B tile + w); it is walked oldest first in chunks of F frames.  Each chunk is
// staged with coalesced 8-byte loads along every channel's row into the bit-reversed slots of one
// row of M + 1 frames per window frame (the padding keeps the loads of a column of rows
// conflict-free), the log2 M stages run in place with a barrier after each, and every output then
// adds the chunk's frames of its own window, w = j + hp - 1 - p, in increasing w.  The chunks keep
// the order of step 2, so the sums are those of one pass; they keep shared memory bounded when hp is
// large.  Consecutive threads take consecutive outputs: their columns n mod M are consecutive, and
// the stores are contiguous.  The stages repeat chan_apply_kernel's loop instead of sharing a helper
// with it: factored into one, that kernel compiles to different code.
__global__ void __launch_bounds__(1024) chan_synth_kernel(const __grid_constant__ ChanSynthCall a)
{
    extern __shared__ __align__(16) float2 sm[];
    const uint32_t tid = threadIdx.x, nthreads = blockDim.x;
    const uint64_t stream = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;
    const uint32_t M = a.m, D = 1u << a.log2up, hn = a.hp - 1, F = a.chunk, stride = M + 1;
    const uint64_t f0 = tile * a.frames;
    const uint32_t nf = uint32_t(min(uint64_t(a.frames), a.nin - f0)); // the tile's input frames
    const uint32_t wlen = nf + hn, nout = nf << a.log2up;
    const float2 *hist = a.hist + stream * M * hn;
    const float2 *in = a.in + stream * M * a.nin;

    float acc_re[kChanSynthBlock], acc_im[kChanSynthBlock];
#pragma unroll
    for (int i = 0; i < kChanSynthBlock; i++)
        acc_re[i] = acc_im[i] = 0.0f;

    for (uint32_t w0 = 0; w0 < wlen; w0 += F) {
        const uint32_t nc = min(F, wlen - w0);
        for (uint32_t e = tid; e < nc * M; e += nthreads) {
            const uint32_t k = e / nc, f = e - k * nc;
            const uint64_t b = f0 + w0 + f; // buffer frame
            const float2 v = b < hn ? hist[uint64_t(k) * hn + b] : in[uint64_t(k) * a.nin + (b - hn)];
            sm[f * stride + (__brev(k) >> (32 - a.log2m))] = v;
        }
        __syncthreads();

        const uint32_t half = M >> 1, nbf = nc * half;
        for (uint32_t s = 0; s < a.log2m; s++) {
            const uint32_t hs = 1u << s;
            for (uint32_t b = tid; b < nbf; b += nthreads) {
                const uint32_t f = b >> (a.log2m - 1), bb = b & (half - 1), jj = bb & (hs - 1);
                float2 *pa = sm + f * stride + ((bb >> s) << (s + 1)) + jj;
                const float2 w = __ldg(a.tw + (jj << (9 - s)));
                const float2 p = pa[0], q = pa[hs];
                const float tr = __fsub_rn(__fmul_rn(q.x, w.x), __fmul_rn(q.y, w.y));
                const float ti = __fadd_rn(__fmul_rn(q.x, w.y), __fmul_rn(q.y, w.x));
                pa[0] = make_float2(__fadd_rn(p.x, tr), __fadd_rn(p.y, ti));
                pa[hs] = make_float2(__fsub_rn(p.x, tr), __fsub_rn(p.y, ti));
            }
            __syncthreads();
        }

#pragma unroll
        for (int i = 0; i < kChanSynthBlock; i++) {
            const uint32_t l = tid + i * nthreads;
            if (l >= nout)
                continue;
            const uint32_t j = l >> a.log2up, t = l & (D - 1);
            const uint32_t np = t < a.ntaps ? (a.ntaps - t + D - 1) >> a.log2up : 0;
            const uint32_t col = uint32_t((a.rot0 + (uint64_t(tile) * a.frames << a.log2up) + l) & (M - 1));
            // frames j + hp - np .. j + hp - 1 of the window, those of this chunk
            const uint32_t lo = max(w0, j + a.hp - np), hi = min(w0 + nc, j + a.hp);
            const float2 *y = sm + col - w0 * stride;
            const float *h = a.taps + t + (j + hn) * D;
            for (uint32_t w = lo; w < hi; w++) {
                const float2 v = y[w * stride];
                const float hv = __ldg(h - w * D);
                acc_re[i] = __fadd_rn(acc_re[i], __fmul_rn(v.x, hv));
                acc_im[i] = __fadd_rn(acc_im[i], __fmul_rn(v.y, hv));
            }
        }
        __syncthreads();
    }

    float2 *out = a.out + stream * (a.nin << a.log2up) + (f0 << a.log2up);
#pragma unroll
    for (int i = 0; i < kChanSynthBlock; i++) {
        const uint32_t l = tid + i * nthreads;
        if (l < nout)
            out[l] = make_float2(acc_re[i], acc_im[i]);
    }
}

} // namespace sx
