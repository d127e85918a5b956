// sx_nco.cuh -- numerically controlled oscillators for streams: each stream's frames multiplied by
// e^{+j 2 pi phi_k / 2^32}, with a 32-bit phase phi_s and a 32-bit increment inc_s per stream kept in
// device memory (tests/sxnco.py restates it in numpy).  Frame k of a call sees the phase
// phi_s + (k mod 2^32) inc_s (mod 2^32), and a call of n frames advances phi_s by n inc_s.
//
// The phasor of a phase is a two-table lookup rounded to 20 bits: u = (phi + 2048) >> 12 (mod 2^32
// before the shift), A[u >> 10] e^{j 2 pi hi / 1024} and B[u & 1023] e^{j 2 pi lo / 2^20}, each
// entry the float32 rounding of libm's double cos / sin (built on the host, sxgpu_nco_create).
//     c = A.re B.re - A.im B.im      s = A.im B.re + A.re B.im
//     y.re = x.re c - x.im s          y.im = x.re s + x.im c
// every product and sum one correctly rounded float32 operation (__fmul_rn / __fadd_rn /
// __fsub_rn, never an FFMA), as in sx_fir.cuh.  The phasor is within 3.1e-6 of e^{j 2 pi phi / 2^32};
// the phase error of the rounding to 20 bits is at most pi 2^-20 rad.
//
// The tables (16 KB) are read through L1; the kernels that stream frames bypass it
// (ld_stream / st_stream), so the tables stay there.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "sx_kernels.cuh"

namespace sx {

constexpr int kNcoTableSize = 1024; // entries of each table: A[0..1023] then B[0..1023]

// What the kernels need of an NCO: its tables and its per-stream state.
struct NcoView {
    const float2 *tab; // [2 kNcoTableSize]: A, then B
    uint32_t *phase;   // [nstreams]
    uint32_t *inc;     // [nstreams]
};

__device__ __forceinline__ float2 nco_phasor(const float2 *tab, uint32_t phi)
{
    const uint32_t u = (phi + 2048u) >> 12;
    const float2 a = __ldg(tab + (u >> 10)), b = __ldg(tab + kNcoTableSize + (u & (kNcoTableSize - 1)));
    return make_float2(__fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)),
                       __fadd_rn(__fmul_rn(a.y, b.x), __fmul_rn(a.x, b.y)));
}

__device__ __forceinline__ float2 nco_mix(float2 x, float2 p)
{
    return make_float2(__fsub_rn(__fmul_rn(x.x, p.x), __fmul_rn(x.y, p.y)),
                       __fadd_rn(__fmul_rn(x.x, p.y), __fmul_rn(x.y, p.x)));
}

// One stream's oscillator for the frames of one call: mix(k, x) is frame k of the call mixed.
struct NcoStream {
    const float2 *tab;
    uint32_t phase, inc;
    __device__ __forceinline__ float2 operator()(uint64_t k, float2 x) const
    {
        return nco_mix(x, nco_phasor(tab, phase + uint32_t(k) * inc));
    }
};

// The oscillator of stream s as the call found it.  A kernel that reads it must end before the
// phase advances (nco_advance, in a later launch or after a barrier of the reading CTA).
__device__ __forceinline__ NcoStream nco_stream(const NcoView &v, uint64_t s)
{
    return NcoStream{v.tab, v.phase[s], v.inc[s]};
}

// Stream s after a call of `frames` frames (mod 2^32).
__device__ __forceinline__ void nco_advance(const NcoView &v, uint64_t s, uint32_t frames)
{
    v.phase[s] += frames * v.inc[s];
}

// No oscillator.  The FIR kernels that can mix (fir_history_kernel, bank_fir_kernel,
// bank_fir_read_tail_kernel) take the oscillator as a template parameter: with NoNco the two
// overloads below compile to nothing, so those instantiations are the plain kernels, and with
// NcoView they are the mixing ones, from the same source.
struct NoNco {
};

struct NoMix {
    __device__ __forceinline__ float2 operator()(uint64_t, float2 x) const { return x; }
};

__device__ __forceinline__ NoMix nco_stream(NoNco, uint64_t) { return {}; }

__device__ __forceinline__ void nco_advance(NoNco, uint64_t, uint32_t) {}

// sxgpu_nco_apply: x[nstreams][nframes] mixed in place, one tile of kNcoTile frames of the flat
// block per CTA, kNcoFramesPerThread frames per thread, kNcoThreads apart so that each warp access
// is 256 contiguous bytes.  A frame's stream is g div nframes, found with a double reciprocal
// (g < 2^41 frames: the grid has fewer than 2^31 CTAs, so g and the quotient's error fit a double's
// mantissa) and corrected by one either way.
constexpr int kNcoThreads = 256, kNcoFramesPerThread = 4, kNcoTile = kNcoThreads * kNcoFramesPerThread;

__global__ void __launch_bounds__(kNcoThreads) nco_apply_kernel(NcoView v, float2 *x, uint64_t nframes, uint64_t total,
                                                                double inv_nframes)
{
    const uint64_t g0 = uint64_t(blockIdx.x) * kNcoTile + threadIdx.x;
    Pack<2> f[kNcoFramesPerThread];
#pragma unroll
    for (int j = 0; j < kNcoFramesPerThread; j++)
        if (g0 + j * kNcoThreads < total)
            f[j] = ld_stream<8>(x + g0 + j * kNcoThreads);
#pragma unroll
    for (int j = 0; j < kNcoFramesPerThread; j++) {
        const uint64_t g = g0 + j * kNcoThreads;
        if (g >= total)
            break;
        uint64_t s = uint64_t(__dmul_rn(__ull2double_rn(g), inv_nframes));
        const int64_t r = int64_t(g - s * nframes);
        if (r < 0)
            s--;
        else if (uint64_t(r) >= nframes)
            s++;
        const float2 y = nco_stream(v, s)(g - s * nframes, make_float2(__uint_as_float(f[j].w[0]), __uint_as_float(f[j].w[1])));
        Pack<2> w;
        w.w[0] = __float_as_uint(y.x), w.w[1] = __float_as_uint(y.y);
        st_stream<8>(x + g, w);
    }
}

// The phases after sxgpu_nco_apply's frames, a launch of its own after every read of the old ones.
__global__ void nco_advance_kernel(NcoView v, uint32_t nstreams, uint32_t frames)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < nstreams)
        nco_advance(v, s, frames);
}

} // namespace sx
