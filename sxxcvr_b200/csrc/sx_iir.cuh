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

// ---- long blocks: chunks, and the float64 carry between them (sxgpu_iir_apply_long) ------------
//
// A block of nstreams x nframes frames is cut into chunks of L frames (the last of a stream may be
// shorter), K = ceil(nframes / L) per stream.  Over a chunk the cascade is linear in its state:
// end = M start + e, M = A^L, with A the 2S x 2S one-step state matrix of the cascade (S sections;
// state index 2 q + j for z_j of section q; built on the host in float64 from the float32
// coefficients, column by column, by one step of the float64 recurrence on zero input).  Then
//     pass 1   every chunk but a stream's last, from a zero state in float32: its end state e_k only
//     carry    per stream and component, in float64, v_0 = zi and v_k = e_{k-1} (k >= 1):
//              s_0 = v_0 and s_k = M s_{k-1} + v_k
//     pass 3   every chunk from float32(s_k), in place; a stream's last chunk leaves the filter state.
// Chunk 0 starts from zi exactly, so its frames are sxgpu_iir_apply's bit for bit.
//
// The carry's evaluation order, which tests/sxiir_long.py restates: every product and sum is one
// correctly rounded float64 operation (__dmul_rn / __dadd_rn), a matrix-vector product is
//     (P x)_i = P_i0 x_0 + P_i1 x_1 + ... + P_i,n-1 x_n-1    (left to right),
// and a step is (P x) + v.  P_j = A^(2^j) by repeated squaring (P_0 = A, P_j+1 = P_j P_j, each
// entry of a matrix product summed the same way), so M = P_log2(L).  Elements go in groups of
// kIirGroup consecutive chunks:
//     reduce   T_g = v_64g; then T_g = M T_g + v_k for the group's later elements, in order
//     scan     W_g = T_g; for d = 1, 2, 4, ... < G (groups per stream): W_g = P_log2(L)+6+log2(d) W_g-d + W_g
//              for g >= d (Hillis-Steele, each level from the previous level's values)
//     fix-up   s_64g = v_0 (g = 0) or M W_g-1 + v_64g, then s_k = M s_k-1 + v_k through the group.
constexpr int kIirDim = 2 * kIirMaxSections; // the state of one component
constexpr int kIirGroup = 64, kIirLog2Group = 6;
constexpr int kIirPowers = 64; // P_0 .. P_63: enough for any exponent L 64 d < 2 nframes < 2^64

// Row layouts of iir_apply_kernel: a row per stream (sxgpu_iir_apply, its state carried in f.state),
// or a row per chunk of a long block, for pass 1 or pass 3.
enum { kIirRowsStreams = 0, kIirRowsChunkEnds = 1, kIirRowsChunkOut = 2 };

// A long block's chunks.  edge: [stream][chunk][component][kIirDim] float32: pass 1 writes chunk k's
// end state to slot k + 1, the fix-up writes chunk k's start state to slot k, which pass 3 reads.
struct IirChunks {
    uint64_t nframes;    // frames per stream
    uint64_t per_stream; // chunks per stream, K
    uint64_t rows;       // rows of the pass: nstreams (K - 1) for pass 1, nstreams K for pass 3
    uint32_t len;        // L
    float *edge;
};

__device__ __forceinline__ float *iir_edge_at(const IirChunks &ch, uint64_t stream, uint64_t k, uint32_t c)
{
    return ch.edge + ((stream * ch.per_stream + k) * 2 + c) * kIirDim;
}

// d_cf32 filtered in place a tile at a time.  A CTA takes kIirStreamsPerCta rows through their
// frames: a coalesced load of the tile (a warp reads 32 consecutive frames of one row), the
// sequential pass, a coalesced store.  Frame-wide accesses, so any length and any 8-byte aligned
// block.  kIirRowsStreams is sxgpu_iir_apply: d_cf32[nstreams][period], the state carried.  The
// chunk layouts take row r as chunk k of stream s (pass 1: r = s (K - 1) + k, pass 3: r = s K + k);
// pass 1 starts from zero and stores no samples.
template <int ROWS = kIirRowsStreams>
__global__ void __launch_bounds__(kIirThreads) iir_apply_kernel(const __grid_constant__ IirView f, char *cf32, uint32_t period,
                                                                const __grid_constant__ IirChunks ch)
{
    __shared__ __align__(16) float tile[kIirStreamsPerCta * kIirRow];
    const uint32_t j = threadIdx.x >> 1, c = threadIdx.x & 1;
    const uint64_t s0 = uint64_t(blockIdx.x) * kIirStreamsPerCta, s = s0 + j;
    if constexpr (ROWS == kIirRowsStreams) {
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
    } else {
        float z[kIirMaxSections][2], none[kIirMaxSections][2];
        IirCoeffs nothing;
        nothing.nsections = 0;
        __shared__ uint64_t row_base[kIirStreamsPerCta]; // first frame of the row in the block
        __shared__ uint32_t row_len[kIirStreamsPerCta];
        const uint32_t count = uint32_t(ch.rows - s0 < kIirStreamsPerCta ? ch.rows - s0 : kIirStreamsPerCta);
        const bool active = j < count;
        const uint64_t chunks = ROWS == kIirRowsChunkEnds ? ch.per_stream - 1 : ch.per_stream;
        const uint64_t stream = s / chunks, k = s % chunks;
        const uint64_t first = k * ch.len;
        const uint32_t len = uint32_t(ch.nframes - first < ch.len ? ch.nframes - first : ch.len);
        if (c == 0 && active) {
            row_base[j] = stream * ch.nframes + first;
            row_len[j] = len;
        }
#pragma unroll
        for (int q = 0; q < kIirMaxSections; q++) {
            const bool on = ROWS == kIirRowsChunkOut && active && q < int(f.k.nsections);
            z[q][0] = on ? iir_edge_at(ch, stream, k, c)[2 * q] : 0.0f;
            z[q][1] = on ? iir_edge_at(ch, stream, k, c)[2 * q + 1] : 0.0f;
        }
        __syncthreads();
        for (uint32_t t0 = 0; t0 < ch.len; t0 += kIirTile) {
            for (uint32_t q = threadIdx.x; q < count * kIirTile; q += kIirThreads) {
                const uint32_t r = q / kIirTile, i = q % kIirTile;
                if (t0 + i < row_len[r])
                    *reinterpret_cast<Pack<2> *>(&tile[r * kIirRow + 2 * i]) = ld_stream<8>(cf32 + (row_base[r] + t0 + i) * 8);
            }
            __syncthreads();
            const uint32_t n = len > t0 ? (len - t0 < kIirTile ? len - t0 : kIirTile) : 0;
            iir_tile_pass<1>(&tile[j * kIirRow], c, n, f.k, z, nothing, none, NoIirHook(), s, active, t0);
            __syncthreads();
            if constexpr (ROWS == kIirRowsChunkOut) {
                for (uint32_t q = threadIdx.x; q < count * kIirTile; q += kIirThreads) {
                    const uint32_t r = q / kIirTile, i = q % kIirTile;
                    if (t0 + i < row_len[r])
                        st_stream<8>(cf32 + (row_base[r] + t0 + i) * 8, *reinterpret_cast<const Pack<2> *>(&tile[r * kIirRow + 2 * i]));
                }
                __syncthreads();
            }
        }
        if constexpr (ROWS == kIirRowsChunkEnds) {
#pragma unroll
            for (int q = 0; q < kIirMaxSections; q++) {
                if (active && q < int(f.k.nsections)) {
                    iir_edge_at(ch, stream, k + 1, c)[2 * q] = z[q][0];
                    iir_edge_at(ch, stream, k + 1, c)[2 * q + 1] = z[q][1];
                }
            }
        } else {
            iir_store_state(f, stream, c, active && k + 1 == ch.per_stream, z);
        }
    }
}

// The carry kernels: a half-warp per (stream, group, component) sequence, lane i holding row i of
// the state and of the matrices.  Sequence q = (stream G + g) 2 + c.
struct IirCarry {
    const double *pow; // [kIirPowers][kIirDim][kIirDim]: P_j, zero outside the 2S x 2S corner
    IirChunks ch;
    const double *in;  // [sequence][kIirDim] group totals: the scan level's input, the fix-up's W
    double *out;       // the reduce's and the scan level's output
    uint64_t groups;   // G
    uint64_t sequences;
    uint32_t log2_len;
};

__device__ __forceinline__ void iir_matrix_row(const IirCarry &a, int j, uint32_t i, double (&p)[kIirDim])
{
#pragma unroll
    for (int col = 0; col < kIirDim; col++)
        p[col] = a.pow[(size_t(j) * kIirDim + i) * kIirDim + col];
}

// (P x)_i, x spread over the half-warp (lane i holds x_i), n = 2S columns, summed left to right.
__device__ __forceinline__ double iir_matvec(const double (&p)[kIirDim], double x, uint32_t n, unsigned mask)
{
    double acc = __dmul_rn(p[0], __shfl_sync(mask, x, 0, 16));
#pragma unroll
    for (int col = 1; col < kIirDim; col++) {
        const double xc = __shfl_sync(mask, x, col, 16);
        if (col < int(n))
            acc = __dadd_rn(acc, __dmul_rn(p[col], xc));
    }
    return acc;
}

// v_k of one stream and component, row i: zi for k = 0, else the edge slot k.
__device__ __forceinline__ double iir_carry_input(const IirView &f, const IirChunks &ch, uint64_t stream, uint64_t k,
                                                  uint32_t c, uint32_t i)
{
    if (i >= 2 * f.k.nsections)
        return 0.0;
    return k == 0 ? double(*iir_state_at(f, int(i >> 1), stream, int(i & 1), c)) : double(iir_edge_at(ch, stream, k, c)[i]);
}

struct IirSequence {
    uint64_t q, stream, g, k0, k1; // chunks [k0, k1) of the group
    uint32_t c, i;
    unsigned mask;
};

__device__ __forceinline__ bool iir_sequence(const IirCarry &a, IirSequence &t)
{
    const uint64_t id = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    t.q = id / 16;
    t.i = uint32_t(id % 16);
    t.mask = 0xffffu << (threadIdx.x & 16);
    if (t.q >= a.sequences)
        return false; // the whole half-warp
    t.c = uint32_t(t.q & 1);
    t.stream = (t.q >> 1) / a.groups;
    t.g = (t.q >> 1) % a.groups;
    t.k0 = t.g * kIirGroup;
    t.k1 = t.k0 + kIirGroup < a.ch.per_stream ? t.k0 + kIirGroup : a.ch.per_stream;
    return true;
}

// Reduce: the group totals T_g into a.out.
__global__ void __launch_bounds__(128) iir_carry_reduce_kernel(const __grid_constant__ IirView f, const __grid_constant__ IirCarry a)
{
    IirSequence t;
    if (!iir_sequence(a, t))
        return;
    const uint32_t n = 2 * f.k.nsections;
    double m[kIirDim];
    iir_matrix_row(a, int(a.log2_len), t.i, m);
    double x = iir_carry_input(f, a.ch, t.stream, t.k0, t.c, t.i);
    for (uint64_t k = t.k0 + 1; k < t.k1; k++)
        x = __dadd_rn(iir_matvec(m, x, n, t.mask), iir_carry_input(f, a.ch, t.stream, k, t.c, t.i));
    a.out[t.q * kIirDim + t.i] = x;
}

// One Hillis-Steele level over the group totals of each stream, groups d = 2^level apart.
__global__ void __launch_bounds__(128) iir_carry_scan_kernel(const __grid_constant__ IirView f, const __grid_constant__ IirCarry a,
                                                             uint32_t level)
{
    IirSequence t;
    if (!iir_sequence(a, t))
        return;
    const uint64_t d = uint64_t(1) << level;
    double x = a.in[t.q * kIirDim + t.i];
    if (t.g >= d) {
        double p[kIirDim];
        iir_matrix_row(a, int(a.log2_len + kIirLog2Group + level), t.i, p);
        x = __dadd_rn(iir_matvec(p, a.in[(t.q - 2 * d) * kIirDim + t.i], 2 * f.k.nsections, t.mask), x);
    }
    a.out[t.q * kIirDim + t.i] = x;
}

// Fix-up: every chunk's start state s_k, rounded to float32, into its edge slot (in place of v_k).
__global__ void __launch_bounds__(128) iir_carry_fixup_kernel(const __grid_constant__ IirView f, const __grid_constant__ IirCarry a)
{
    IirSequence t;
    if (!iir_sequence(a, t))
        return;
    const uint32_t n = 2 * f.k.nsections;
    double m[kIirDim];
    iir_matrix_row(a, int(a.log2_len), t.i, m);
    double x = iir_carry_input(f, a.ch, t.stream, t.k0, t.c, t.i);
    if (t.g > 0)
        x = __dadd_rn(iir_matvec(m, a.in[(t.q - 2) * kIirDim + t.i], n, t.mask), x);
    for (uint64_t k = t.k0;;) {
        if (t.i < n)
            iir_edge_at(a.ch, t.stream, k, t.c)[t.i] = __double2float_rn(x);
        if (++k >= t.k1)
            break;
        x = __dadd_rn(iir_matvec(m, x, n, t.mask), iir_carry_input(f, a.ch, t.stream, k, t.c, t.i));
    }
}

} // namespace sx
