// sx_iir.cuh -- stateful IIR filters for a bank of streams: cascaded second-order sections in
// scipy's transposed direct form II, with real float32 coefficients, applied to the I and the Q
// component of CF32 samples independently (what scipy.signal.sosfilt does with a real `sos` on
// complex input).  The reference repeater filters its blocks with such a channel filter before
// and after its clipper (example/linear_repeater.py:78-109), carrying the state from block to block.
//
// A recurrence along one stream is sequential, but a bank has thousands of streams: one lane per
// (stream, component) runs the cascade over the period with the state in registers, reading the
// state once at the start and writing it once at the end.  Samples reach the lanes through
// shared memory, so that global loads and stores stay coalesced (tiles of kIirTile frames of
// kIirStreamsPerCta streams: a row per stream, component c of frame i at row[2 * i + c]).
//
// Rounding.  For one sample x of one component and one section, in exactly this order, every
// operation one correctly rounded float32 operation (the _rn intrinsics are never contracted into
// an FMA; the build keeps denormals, so decaying state ends in subnormals as it does on a CPU):
//     y  = b0*x + z0
//     z0 = (b1*x - a1*y) + z1
//     z1 = b2*x - a2*y
// which is scipy's own loop (scipy/signal/_sosfilt.pyx) on float32, and gives the same bits as
// sosfilt on complex64 input with float32 coefficients (tests/sxiir.py restates it in numpy).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "sx_kernels.cuh"

namespace sx {

constexpr int kIirMaxSections = 8; // SXGPU_IIR_MAX_SECTIONS: order 16

// The coefficients of one cascade, rounded from the caller's float64 to float32 once, on the host.
// a0 is 1 (checked on the host) and not stored.  Passed to kernels as a __grid_constant__
// parameter: every stream of a filter shares them, so they are uniform operands, not loads.
struct IirCoeffs {
    float b0[kIirMaxSections], b1[kIirMaxSections], b2[kIirMaxSections];
    float a1[kIirMaxSections], a2[kIirMaxSections];
    uint32_t nsections; // 0: no filter (a stage of the fused iteration left out)
};

// One filter of a bank as the kernels see it (sxgpu_iir_device_view hands it to sx_hook.cuh).
struct IirView {
    uint32_t nstreams;
    float *state; // [nsections][nstreams][2: z0, z1][2: I, Q] -- scipy's zi layout for (nstreams, n) input
    IirCoeffs k;
};

__device__ __forceinline__ void iir_section(float &x, float &z0, float &z1, float b0, float b1, float b2, float a1, float a2)
{
    const float y = __fadd_rn(__fmul_rn(b0, x), z0);
    z0 = __fadd_rn(__fsub_rn(__fmul_rn(b1, x), __fmul_rn(a1, y)), z1);
    z1 = __fsub_rn(__fmul_rn(b2, x), __fmul_rn(a2, y));
    x = y;
}

// F consecutive samples of one component through the whole cascade, section by section: section q
// takes all F before section q + 1 starts, so the test on the (uniform) section count is taken
// once per F samples, and the state stays in registers under static indices.
template <int F>
__device__ __forceinline__ void iir_cascade(const IirCoeffs &k, float (&z)[kIirMaxSections][2], float (&x)[F])
{
#pragma unroll
    for (int q = 0; q < kIirMaxSections; q++) {
        if (q >= int(k.nsections))
            break;
#pragma unroll
        for (int i = 0; i < F; i++)
            iir_section(x[i], z[q][0], z[q][1], k.b0[q], k.b1[q], k.b2[q], k.a1[q], k.a2[q]);
    }
}

__device__ __forceinline__ float *iir_state_at(const IirView &f, int q, uint64_t s, int j, uint32_t c)
{
    return f.state + ((uint64_t(q) * f.nstreams + s) * 2 + j) * 2 + c;
}

__device__ __forceinline__ void iir_load_state(const IirView &f, uint64_t s, uint32_t c, bool active,
                                               float (&z)[kIirMaxSections][2])
{
#pragma unroll
    for (int q = 0; q < kIirMaxSections; q++) {
        const bool on = active && q < int(f.k.nsections);
        z[q][0] = on ? *iir_state_at(f, q, s, 0, c) : 0.0f;
        z[q][1] = on ? *iir_state_at(f, q, s, 1, c) : 0.0f;
    }
}

__device__ __forceinline__ void iir_store_state(const IirView &f, uint64_t s, uint32_t c, bool active,
                                                const float (&z)[kIirMaxSections][2])
{
#pragma unroll
    for (int q = 0; q < kIirMaxSections; q++) {
        if (active && q < int(f.k.nsections)) {
            *iir_state_at(f, q, s, 0, c) = z[q][0];
            *iir_state_at(f, q, s, 1, c) = z[q][1];
        }
    }
}

// Tiles through shared memory: kIirStreamsPerCta streams (two lanes each) x kIirTile frames.  A
// row holds one stream's tile; its length is padded by four floats so that the sixteen streams of
// a warp in the sequential pass fall on different banks (two-way at worst) while rows stay
// 16-byte aligned for the vector stores of the coalesced passes.
constexpr int kIirStreamsPerCta = 64, kIirThreads = 2 * kIirStreamsPerCta, kIirTile = 32, kIirRow = 2 * kIirTile + 4;

// The memoryless stage between the two cascades (sx_hook.cuh): identity unless a functor is given.
struct NoIirHook {};

// The sequential pass over one tile, in place: lane 2 j + c takes component c of the row of
// stream s = (first stream of the CTA) + j, frames [0, n) of the tile, which are frames
// [frame0, frame0 + n) of the stream's block: pre cascade, then `hook` on each pair of frames
// (both lanes of the stream evaluate it on the same Pack<4>, and each keeps its component; every
// lane of the warp must get here, with the same n), then post cascade.  With a hook, n is even.
template <int F, class Hook>
__device__ __forceinline__ void iir_tile_chunk(float *row, uint32_t c, uint32_t f0, const IirCoeffs &pre,
                                               float (&zp)[kIirMaxSections][2], const IirCoeffs &post,
                                               float (&zq)[kIirMaxSections][2], const Hook &hook, uint64_t s,
                                               bool active, uint32_t frame0)
{
    float x[F];
#pragma unroll
    for (int i = 0; i < F; i++)
        x[i] = row[2 * (f0 + i) + c];
    iir_cascade<F>(pre, zp, x);
    if constexpr (!std::is_same<Hook, NoIirHook>::value) {
        static_assert(F % 2 == 0, "the hook takes pairs of frames");
#pragma unroll
        for (int p = 0; p < F / 2; p++) {
            const float o0 = __shfl_xor_sync(0xffffffffu, x[2 * p], 1);
            const float o1 = __shfl_xor_sync(0xffffffffu, x[2 * p + 1], 1);
            Pack<4> v;
            v.w[0] = __float_as_uint(c ? o0 : x[2 * p]);
            v.w[1] = __float_as_uint(c ? x[2 * p] : o0);
            v.w[2] = __float_as_uint(c ? o1 : x[2 * p + 1]);
            v.w[3] = __float_as_uint(c ? x[2 * p + 1] : o1);
            if (active)
                hook(v, s, frame0 + f0 + 2 * p);
            x[2 * p] = __uint_as_float(c ? v.w[1] : v.w[0]);
            x[2 * p + 1] = __uint_as_float(c ? v.w[3] : v.w[2]);
        }
    }
    iir_cascade<F>(post, zq, x);
#pragma unroll
    for (int i = 0; i < F; i++)
        row[2 * (f0 + i) + c] = x[i];
}

template <int TAIL, class Hook>
__device__ __forceinline__ void iir_tile_pass(float *row, uint32_t c, uint32_t n, const IirCoeffs &pre,
                                              float (&zp)[kIirMaxSections][2], const IirCoeffs &post,
                                              float (&zq)[kIirMaxSections][2], const Hook &hook, uint64_t s,
                                              bool active, uint32_t frame0)
{
    uint32_t f0 = 0;
    for (; f0 + 8 <= n; f0 += 8)
        iir_tile_chunk<8>(row, c, f0, pre, zp, post, zq, hook, s, active, frame0);
    for (; f0 < n; f0 += TAIL)
        iir_tile_chunk<TAIL>(row, c, f0, pre, zp, post, zq, hook, s, active, frame0);
}

// sxgpu_iir_apply: d_cf32[nstreams][period] filtered in place, the state carried.  A CTA takes
// kIirStreamsPerCta streams through the period tile by tile: a coalesced load of the tile (a warp
// reads 32 consecutive frames of one stream), the sequential pass, a coalesced store.  Frame-wide
// accesses, so any period and any 8-byte aligned block.
__global__ void __launch_bounds__(kIirThreads) iir_apply_kernel(const __grid_constant__ IirView f, char *cf32, uint32_t period)
{
    __shared__ __align__(16) float tile[kIirStreamsPerCta * kIirRow];
    const uint32_t j = threadIdx.x >> 1, c = threadIdx.x & 1;
    const uint64_t s0 = uint64_t(blockIdx.x) * kIirStreamsPerCta, s = s0 + j;
    const uint32_t count = uint32_t(f.nstreams - s0 < kIirStreamsPerCta ? f.nstreams - s0 : kIirStreamsPerCta);
    const bool active = j < count;
    float z[kIirMaxSections][2], none[kIirMaxSections][2];
    iir_load_state(f, s, c, active, z);
    IirCoeffs nothing;
    nothing.nsections = 0;
    for (uint32_t t0 = 0; t0 < period; t0 += kIirTile) {
        const uint32_t n = period - t0 < kIirTile ? period - t0 : kIirTile;
        for (uint32_t q = threadIdx.x; q < count * kIirTile; q += kIirThreads) {
            const uint32_t r = q / kIirTile, i = q % kIirTile;
            if (i < n)
                *reinterpret_cast<Pack<2> *>(&tile[r * kIirRow + 2 * i]) = ld_stream<8>(cf32 + ((s0 + r) * period + t0 + i) * 8);
        }
        __syncthreads();
        iir_tile_pass<1>(&tile[j * kIirRow], c, n, f.k, z, nothing, none, NoIirHook(), s, active, t0);
        __syncthreads();
        for (uint32_t q = threadIdx.x; q < count * kIirTile; q += kIirThreads) {
            const uint32_t r = q / kIirTile, i = q % kIirTile;
            if (i < n)
                st_stream<8>(cf32 + ((s0 + r) * period + t0 + i) * 8, *reinterpret_cast<const Pack<2> *>(&tile[r * kIirRow + 2 * i]));
        }
        __syncthreads(); // the next tile's loads overwrite the rows
    }
    iir_store_state(f, s, c, active, z);
}

} // namespace sx
