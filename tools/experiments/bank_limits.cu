// bank_limits.cu -- what bounds one repeater iteration of the stream bank (BASELINE config 4)?
//
// The fused iteration (sxgpu_bank_repeat) writes three regions per stream and period -- capture
// slot, caller's CF32 block, playback ring: 24 B/frame, 402 MB at 65536 streams x 256 frames --
// and every schedule tried so far lands at 68-76 us.  This program splits that figure at the
// bank's exact shape:
//   memset            cudaMemsetAsync over the same three regions (the write-only ceiling used as
//                     the yardstick in profiles/)
//   store_only        the same bytes by plain 128-/256-bit stores, no arithmetic: cache hints,
//                     CTAs per SM, vectors in flight per lane, 1/2/3 regions
//   fused_flat        the whole arithmetic (synthetic capture, RX, TX conversions) in registers
//                     in front of those stores, per-stream decisions read from two arrays
// Standalone: only the PTX helpers and the conversion ops of sx_kernels.cuh, none of the library.
//     nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I sxxcvr_b200/csrc \
//          -o tools/experiments/bin/bank_limits tools/experiments/bank_limits.cu
// Prints one JSON object per line.  NOT a product path.
#include "sx_bank.cuh"
#include "sx_kernels.cuh"
#include "sx_synth.h"
#include "sx_time.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

using namespace sx;

#define CK(x)                                                                                      \
    do {                                                                                           \
        cudaError_t e_ = (x);                                                                      \
        if (e_ != cudaSuccess) {                                                                   \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_));             \
            exit(1);                                                                               \
        }                                                                                          \
    } while (0)

struct Regions {
    char *slot, *cf, *ring; // [nstreams][period] frames each
    const long long *first; // per stream: counter of its first captured frame
    const long long *at;    // per stream: where its block is written (unused here: lock-step)
    uint32_t nstreams, period;
    uint64_t seed;
    float thr2;
};

template <int HINT> __device__ __forceinline__ void store16(void *p, const Pack<4> &v)
{
    if constexpr (HINT == 0)
        asm volatile("st.global.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
    else if constexpr (HINT == 1)
        asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
    else if constexpr (HINT == 2)
        asm volatile("st.global.cs.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
    else
        asm volatile("st.global.cg.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3]) : "memory");
}

__device__ __forceinline__ void store32(void *p, const Pack<4> &a, const Pack<4> &b)
{
    asm volatile("st.global.L1::no_allocate.L2::evict_first.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(a.w[0]),
                 "r"(a.w[1]), "r"(a.w[2]), "r"(a.w[3]), "r"(b.w[0]), "r"(b.w[1]), "r"(b.w[2]), "r"(b.w[3])
                 : "memory");
}

// Stores only.  A warp takes one stream's period at a time (period / 2 16-byte vectors, U per
// lane in flight), NREG regions.
template <int HINT, int U, int NREG> __global__ void __launch_bounds__(256) store_only_kernel(Regions r)
{
    const uint32_t lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * wpc;
    const uint32_t nvec = r.period / 2;
    for (uint64_t s = uint64_t(blockIdx.x) * wpc + (threadIdx.x >> 5); s < r.nstreams; s += nwarps) {
        const size_t base = s * r.period * 8;
        for (uint32_t b = 0; b < nvec; b += 32 * U) {
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t v = b + lane + 32 * u;
                Pack<4> x;
                x.w[0] = v, x.w[1] = uint32_t(s), x.w[2] = lane, x.w[3] = u;
                if (v < nvec) {
                    store16<HINT>(r.slot + base + size_t(v) * 16, x);
                    if (NREG > 1)
                        store16<HINT>(r.cf + base + size_t(v) * 16, x);
                    if (NREG > 2)
                        store16<HINT>(r.ring + base + size_t(v) * 16, x);
                }
            }
        }
    }
}

// The same bytes by 256-bit stores (32 B per lane, a warp store covers 1 KiB).
template <int U> __global__ void __launch_bounds__(256) store_only256_kernel(Regions r)
{
    const uint32_t lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * wpc;
    const uint32_t nvec = r.period / 4;
    for (uint64_t s = uint64_t(blockIdx.x) * wpc + (threadIdx.x >> 5); s < r.nstreams; s += nwarps) {
        const size_t base = s * r.period * 8;
        for (uint32_t b = 0; b < nvec; b += 32 * U) {
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t v = b + lane + 32 * u;
                Pack<4> x;
                x.w[0] = v, x.w[1] = uint32_t(s), x.w[2] = lane, x.w[3] = u;
                if (v < nvec) {
                    store32(r.slot + base + size_t(v) * 32, x, x);
                    store32(r.cf + base + size_t(v) * 32, x, x);
                    store32(r.ring + base + size_t(v) * 32, x, x);
                }
            }
        }
    }
}

// Stores only, flat: thread t of the grid writes vector t, t + T, ... of each region (a warp's
// store covers 512 contiguous bytes; consecutive warps of a CTA consecutive 512-byte pieces).
template <int HINT, int U> __global__ void __launch_bounds__(256) store_flat_kernel(Regions r)
{
    const uint64_t total = uint64_t(r.nstreams) * r.period / 2, T = uint64_t(gridDim.x) * blockDim.x;
    for (uint64_t v0 = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; v0 < total; v0 += T * U) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = v0 + u * T;
            Pack<4> x;
            x.w[0] = uint32_t(v), x.w[1] = uint32_t(v >> 32), x.w[2] = threadIdx.x, x.w[3] = u;
            if (v < total) {
                store16<HINT>(r.slot + v * 16, x);
                store16<HINT>(r.cf + v * 16, x);
                store16<HINT>(r.ring + v * 16, x);
            }
        }
    }
}

// All of the iteration's arithmetic in registers, then the stores: warp per stream, U vectors
// per lane in flight, decisions (first captured frame) read per stream.
template <int HINT, int U, int MINB, bool WIDE> __global__ void __launch_bounds__(256, MINB) fused_flat_kernel(Regions r)
{
    const uint32_t lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * wpc;
    const uint32_t nvec = r.period / 2;
    for (uint64_t s = uint64_t(blockIdx.x) * wpc + (threadIdx.x >> 5); s < r.nstreams; s += nwarps) {
        const size_t base = s * r.period * 8;
        const uint64_t first = uint64_t(r.first[s]);
        const uint64_t seed = r.seed + s;
        for (uint32_t b = 0; b < nvec; b += 32 * U * (WIDE ? 2 : 1)) {
            Pack<4> cap[U * (WIDE ? 2 : 1)], mid[U * (WIDE ? 2 : 1)], out[U * (WIDE ? 2 : 1)];
            constexpr int N = U * (WIDE ? 2 : 1);
#pragma unroll
            for (int u = 0; u < N; u++) {
                // WIDE: a lane owns pairs of adjacent vectors (32 B), so that its stores are 256-bit
                const uint32_t v = WIDE ? b + 2 * (lane + 32 * (u / 2)) + (u & 1) : b + lane + 32 * u;
                const uint64_t z0 = sx_synth_frame(seed, first + 2 * uint64_t(v));
                const uint64_t z1 = sx_synth_frame(seed, first + 2 * uint64_t(v) + 1);
                cap[u].w[0] = uint32_t(z0), cap[u].w[1] = uint32_t(z0 >> 32);
                cap[u].w[2] = uint32_t(z1), cap[u].w[3] = uint32_t(z1 >> 32);
                RxCf32::apply<2>(cap[u], mid[u], 0.0f);
                TxCf32::apply<2>(mid[u], out[u], r.thr2);
            }
            if constexpr (WIDE) {
#pragma unroll
                for (int u = 0; u < N; u += 2) {
                    const uint32_t v = b + 2 * (lane + 32 * (u / 2));
                    if (v < nvec) {
                        store32(r.slot + base + size_t(v) * 16, cap[u], cap[u + 1]);
                        store32(r.cf + base + size_t(v) * 16, mid[u], mid[u + 1]);
                        store32(r.ring + base + size_t(v) * 16, out[u], out[u + 1]);
                    }
                }
            } else {
#pragma unroll
                for (int u = 0; u < N; u++) {
                    const uint32_t v = b + lane + 32 * u;
                    if (v < nvec) {
                        store16<HINT>(r.slot + base + size_t(v) * 16, cap[u]);
                        store16<HINT>(r.cf + base + size_t(v) * 16, mid[u]);
                        store16<HINT>(r.ring + base + size_t(v) * 16, out[u]);
                    }
                }
            }
        }
    }
}

// The arithmetic alone (one store per warp at the end so that nothing is optimised away).
template <int U> __global__ void __launch_bounds__(256) compute_only_kernel(Regions r)
{
    const uint32_t lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    const uint64_t nwarps = uint64_t(gridDim.x) * wpc;
    const uint32_t nvec = r.period / 2;
    uint32_t acc = 0;
    for (uint64_t s = uint64_t(blockIdx.x) * wpc + (threadIdx.x >> 5); s < r.nstreams; s += nwarps) {
        const uint64_t first = uint64_t(r.first[s]);
        const uint64_t seed = r.seed + s;
        for (uint32_t b = 0; b < nvec; b += 32 * U) {
#pragma unroll
            for (int u = 0; u < U; u++) {
                const uint32_t v = b + lane + 32 * u;
                Pack<4> cap, mid, out;
                const uint64_t z0 = sx_synth_frame(seed, first + 2 * uint64_t(v));
                const uint64_t z1 = sx_synth_frame(seed, first + 2 * uint64_t(v) + 1);
                cap.w[0] = uint32_t(z0), cap.w[1] = uint32_t(z0 >> 32);
                cap.w[2] = uint32_t(z1), cap.w[3] = uint32_t(z1 >> 32);
                RxCf32::apply<2>(cap, mid, 0.0f);
                TxCf32::apply<2>(mid, out, r.thr2);
                acc ^= out.w[0] ^ out.w[1] ^ out.w[2] ^ out.w[3] ^ mid.w[1];
            }
        }
    }
    if (acc == 0x12345678u)
        reinterpret_cast<uint32_t *>(r.slot)[threadIdx.x] = acc;
}


// Stores only, CTA-contiguous chunks: CTA c (of a non-persistent grid, or chunk c of a persistent
// one) writes vectors [c * 256 * U, (c + 1) * 256 * U) of each region, thread t its vectors
// t, t + 256, ... -- the pattern of a one-launch iteration in which a CTA owns whole streams.
template <int HINT, int U, bool PERSISTENT> __global__ void __launch_bounds__(256) store_chunk_kernel(Regions r)
{
    const uint64_t total = uint64_t(r.nstreams) * r.period / 2;
    const uint64_t nchunks = (total + 256 * U - 1) / (256 * U);
    for (uint64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = c * 256 * U + u * 256 + threadIdx.x;
            Pack<4> x;
            x.w[0] = uint32_t(v), x.w[1] = uint32_t(v >> 32), x.w[2] = threadIdx.x, x.w[3] = u;
            if (v < total) {
                store16<HINT>(r.slot + v * 16, x);
                store16<HINT>(r.cf + v * 16, x);
                store16<HINT>(r.ring + v * 16, x);
            }
        }
        if (!PERSISTENT)
            break;
    }
}

// Stores only, flat and non-persistent: one CTA per 256 vectors of each of U far-apart windows.
template <int HINT, int U> __global__ void __launch_bounds__(256) store_flat_np_kernel(Regions r)
{
    const uint64_t total = uint64_t(r.nstreams) * r.period / 2, window = total / U;
    const uint64_t v0 = uint64_t(blockIdx.x) * 256 + threadIdx.x;
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint64_t v = v0 + u * window;
        Pack<4> x;
        x.w[0] = uint32_t(v), x.w[1] = uint32_t(v >> 32), x.w[2] = threadIdx.x, x.w[3] = u;
        if (v0 < window) {
            store16<HINT>(r.slot + v * 16, x);
            store16<HINT>(r.cf + v * 16, x);
            store16<HINT>(r.ring + v * 16, x);
        }
    }
}

// The whole arithmetic in front of the flat pattern: thread t of the grid takes vectors
// t, t + T, ...; the stream a vector belongs to and its place in the period are shifts.
template <int HINT, int U, int MINB> __global__ void __launch_bounds__(256, MINB) fused_grid_flat_kernel(Regions r)
{
    const uint64_t total = uint64_t(r.nstreams) * r.period / 2, T = uint64_t(gridDim.x) * blockDim.x;
    const uint32_t log2v = 31 - __clz(r.period / 2), vmask = r.period / 2 - 1;
    for (uint64_t v0 = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; v0 < total; v0 += T * U) {
        Pack<4> cap[U], mid[U], out[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = v0 + u * T;
            const uint64_t s = v >> log2v;
            const uint32_t k = uint32_t(v) & vmask;
            const uint64_t first = v < total ? uint64_t(__ldg(r.first + s)) : 0;
            const uint64_t z0 = sx_synth_frame(r.seed + s, first + 2 * uint64_t(k));
            const uint64_t z1 = sx_synth_frame(r.seed + s, first + 2 * uint64_t(k) + 1);
            cap[u].w[0] = uint32_t(z0), cap[u].w[1] = uint32_t(z0 >> 32);
            cap[u].w[2] = uint32_t(z1), cap[u].w[3] = uint32_t(z1 >> 32);
            RxCf32::apply<2>(cap[u], mid[u], 0.0f);
            TxCf32::apply<2>(mid[u], out[u], r.thr2);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = v0 + u * T;
            if (v < total) {
                store16<HINT>(r.slot + v * 16, cap[u]);
                store16<HINT>(r.cf + v * 16, mid[u]);
                store16<HINT>(r.ring + v * 16, out[u]);
            }
        }
    }
}

// The same with CTA-contiguous chunks, one chunk per CTA (non-persistent) or a loop of them.
template <int HINT, int U, int MINB, bool PERSISTENT>
__global__ void __launch_bounds__(256, MINB) fused_chunk_kernel(Regions r)
{
    const uint64_t total = uint64_t(r.nstreams) * r.period / 2;
    const uint64_t nchunks = (total + 256 * U - 1) / (256 * U);
    const uint32_t log2v = 31 - __clz(r.period / 2), vmask = r.period / 2 - 1;
    for (uint64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
        Pack<4> cap[U], mid[U], out[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = c * 256 * U + u * 256 + threadIdx.x;
            const uint64_t s = v >> log2v;
            const uint32_t k = uint32_t(v) & vmask;
            const uint64_t first = v < total ? uint64_t(__ldg(r.first + s)) : 0;
            const uint64_t z0 = sx_synth_frame(r.seed + s, first + 2 * uint64_t(k));
            const uint64_t z1 = sx_synth_frame(r.seed + s, first + 2 * uint64_t(k) + 1);
            cap[u].w[0] = uint32_t(z0), cap[u].w[1] = uint32_t(z0 >> 32);
            cap[u].w[2] = uint32_t(z1), cap[u].w[3] = uint32_t(z1 >> 32);
            RxCf32::apply<2>(cap[u], mid[u], 0.0f);
            TxCf32::apply<2>(mid[u], out[u], r.thr2);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const uint64_t v = c * 256 * U + u * 256 + threadIdx.x;
            if (v < total) {
                store16<HINT>(r.slot + v * 16, cap[u]);
                store16<HINT>(r.cf + v * 16, mid[u]);
                store16<HINT>(r.ring + v * 16, out[u]);
            }
        }
        if (!PERSISTENT)
            break;
    }
}


// ---- third pass: do the converters themselves gain from hardware-scheduled (non-persistent)
// CTAs?  One CTA per 256 * U vectors, loads first, then the conversion, then the stores.
struct ConvArgs {
    const char *src;
    char *dst, *dst2;
    uint64_t nvec;
    float thr2;
};
template <class Op, int U, int LHINT> __global__ void __launch_bounds__(256) convert_np_kernel(ConvArgs a)
{
    const uint64_t base = uint64_t(blockIdx.x) * 256 * U + threadIdx.x;
    Pack<4> in[U], out[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * 256 < a.nvec) {
            if (LHINT == 0)
                in[u] = ld_stream<16>(a.src + (base + u * 256) * 16);
            else
                asm volatile("ld.global.nc.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(in[u].w[0]), "=r"(in[u].w[1]), "=r"(in[u].w[2]), "=r"(in[u].w[3])
                             : "l"(a.src + (base + u * 256) * 16));
        }
#pragma unroll
    for (int u = 0; u < U; u++)
        Op::template apply<2>(in[u], out[u], a.thr2);
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * 256 < a.nvec)
            store16<1>(a.dst + (base + u * 256) * 16, out[u]);
}
// the same with each thread's U vectors adjacent (thread-contiguous 16*U bytes)
template <class Op, int U> __global__ void __launch_bounds__(256) convert_np_adjacent_kernel(ConvArgs a)
{
    const uint64_t base = (uint64_t(blockIdx.x) * 256 + threadIdx.x) * U;
    Pack<4> in[U], out[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u < a.nvec)
            in[u] = ld_stream<16>(a.src + (base + u) * 16);
#pragma unroll
    for (int u = 0; u < U; u++)
        Op::template apply<2>(in[u], out[u], a.thr2);
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u < a.nvec)
            store16<1>(a.dst + (base + u) * 16, out[u]);
}
// RX then TX of the same frames, CF32 kept (the fused loopback: 8 R + 8 W + 8 W per frame)
template <int U> __global__ void __launch_bounds__(256) loopback_np_kernel(ConvArgs a)
{
    const uint64_t base = uint64_t(blockIdx.x) * 256 * U + threadIdx.x;
    Pack<4> in[U], mid[U], out[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * 256 < a.nvec)
            in[u] = ld_stream<16>(a.src + (base + u * 256) * 16);
#pragma unroll
    for (int u = 0; u < U; u++) {
        RxCf32::apply<2>(in[u], mid[u], 0.0f);
        TxCf32::apply<2>(mid[u], out[u], a.thr2);
    }
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * 256 < a.nvec) {
            store16<1>(a.dst + (base + u * 256) * 16, mid[u]);
            store16<1>(a.dst2 + (base + u * 256) * 16, out[u]);
        }
}

// ---- the bank iteration with a plan of realistic cost in front: the CTA's first G threads
// each take one stream's decisions (three counters in, double-precision timestamp arithmetic,
// a dozen results out), hand them over in shared memory, then all threads move the samples.
struct PlanArrays {
    long long *clock, *rx_pos, *tx_pos, *rx_time, *first, *at, *gap, *start;
    int *rx_ret, *rx_flags, *tx_ret;
    double rate;
};
template <int U, int BLOCK, bool EXTERNAL> __global__ void __launch_bounds__(BLOCK) bank_np_kernel(Regions r, PlanArrays p)
{
    constexpr int VPC = BLOCK * U;        // vectors per CTA
    const uint32_t nvec = r.period / 2;   // per stream (a power of two here)
    const uint32_t log2v = 31 - __clz(nvec);
    const uint32_t G = VPC >> log2v;      // streams per CTA
    __shared__ long long s_first[64], s_at[64];
    const uint64_t s0 = uint64_t(blockIdx.x) * G;
    if (threadIdx.x < G && s0 + threadIdx.x < r.nstreams) {
        const uint64_t s = s0 + threadIdx.x;
        long long clock = p.clock[s], rx = p.rx_pos[s], tx = p.tx_pos[s];
        long pending = long(clock - rx);
        if (pending < long(r.period))
            clock += long(r.period) - pending;
        const long long t_ns = sx_ticks_to_time_ns(rx, p.rate);
        const long long ticks = sx_time_ns_to_ticks(t_ns + 10240000, p.rate);
        long long at = ticks > tx ? ticks : tx;
        long long gap = at - tx;
        if (at < clock)
            at = -1;
        p.rx_time[s] = t_ns, p.rx_flags[s] = 4, p.first[s] = rx, p.rx_ret[s] = int(r.period);
        p.rx_pos[s] = rx + r.period, p.gap[s] = gap, p.start[s] = tx, p.at[s] = at, p.tx_ret[s] = int(r.period);
        p.tx_pos[s] = (at < 0 ? tx : at) + r.period, p.clock[s] = clock;
        s_first[threadIdx.x] = rx;
        s_at[threadIdx.x] = at;
    }
    __syncthreads();
    const uint64_t vbase = s0 << log2v;
    const uint64_t total = uint64_t(r.nstreams) << log2v;
    Pack<4> cap[U], mid[U], out[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint32_t idx = u * BLOCK + threadIdx.x;
        const uint32_t j = idx >> log2v, k = idx & (nvec - 1);
        const uint64_t v = vbase + idx;
        if (EXTERNAL) {
            if (v < total)
                cap[u] = ld_stream<16>(r.slot + v * 16);
        } else {
            const uint64_t first = uint64_t(s_first[j]);
            const uint64_t z0 = sx_synth_frame(r.seed + s0 + j, first + 2 * uint64_t(k));
            const uint64_t z1 = sx_synth_frame(r.seed + s0 + j, first + 2 * uint64_t(k) + 1);
            cap[u].w[0] = uint32_t(z0), cap[u].w[1] = uint32_t(z0 >> 32);
            cap[u].w[2] = uint32_t(z1), cap[u].w[3] = uint32_t(z1 >> 32);
        }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
        RxCf32::apply<2>(cap[u], mid[u], 0.0f);
        TxCf32::apply<2>(mid[u], out[u], r.thr2);
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
        const uint32_t idx = u * BLOCK + threadIdx.x;
        const uint32_t j = idx >> log2v;
        const uint64_t v = vbase + idx;
        if (v < total) {
            if (!EXTERNAL)
                store16<1>(r.slot + v * 16, cap[u]);
            store16<1>(r.cf + v * 16, mid[u]);
            if (s_at[j] >= 0)
                store16<1>(r.ring + v * 16, out[u]);
        }
    }
}


// ---- fourth pass: the shape of the hardware-scheduled converter: block size, vectors per
// thread, 128- or 256-bit accesses, cache hints.
template <int SH> __device__ __forceinline__ void store32h(void *p, const Pack<8> &v)
{
    if constexpr (SH == 0)
        asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]),
                     "r"(v.w[3]), "r"(v.w[4]), "r"(v.w[5]), "r"(v.w[6]), "r"(v.w[7])
                     : "memory");
    else
        st_stream<32>(p, v);
}
template <class Op, int U, int BLOCK, int W, int SH> __global__ void __launch_bounds__(BLOCK) convert_np2_kernel(ConvArgs a)
{
    // a.nvec counts 16-byte vectors; W = bytes per access
    constexpr int FR = W / 8;
    const uint64_t nacc = a.nvec * 16 / W;
    const uint64_t base = uint64_t(blockIdx.x) * BLOCK * U + threadIdx.x;
    Pack<W / 4> in[U], out[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * BLOCK < nacc)
            in[u] = ld_stream<W>(a.src + (base + u * BLOCK) * W);
#pragma unroll
    for (int u = 0; u < U; u++)
        Op::template apply<FR>(in[u], out[u], a.thr2);
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * BLOCK < nacc) {
            if constexpr (W == 16)
                store16<SH>(a.dst + (base + u * BLOCK) * W, out[u]);
            else
                store32h<SH>(a.dst + (base + u * BLOCK) * W, out[u]);
        }
}
// 12 B/frame extension shapes: 4 frames per thread access, 32 B in / 16 B out (RX CS16) or the reverse
template <class Op, int U, int BLOCK> __global__ void __launch_bounds__(BLOCK) convert_np_narrow_kernel(ConvArgs a)
{
    constexpr int FR = 4, SB = Op::kSrcWords * 4 * FR, DB = Op::kDstWords * 4 * FR;
    const uint64_t nacc = a.nvec / 2; // groups of four frames
    const uint64_t base = uint64_t(blockIdx.x) * BLOCK * U + threadIdx.x;
    Pack<SB / 4> in[U];
    Pack<DB / 4> out[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * BLOCK < nacc)
            in[u] = ld_stream<SB>(a.src + (base + u * BLOCK) * SB);
#pragma unroll
    for (int u = 0; u < U; u++)
        Op::template apply<FR>(in[u], out[u], a.thr2);
#pragma unroll
    for (int u = 0; u < U; u++)
        if (base + u * BLOCK < nacc)
            st_stream<DB>(a.dst + (base + u * BLOCK) * DB, out[u]);
}

static int g_sms = 148;
static cudaEvent_t e0, e1;
constexpr int kSlices = 4;

template <class F> static double time_us(F &&launch, int reps = 30)
{
    for (int i = 0; i < 3; i++)
        launch(i);
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; i++)
        launch(i);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaGetLastError());
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    return double(ms) * 1e3 / reps;
}

static void report(const std::string &name, double us, double bytes)
{
    printf("{\"kernel\": \"%s\", \"us\": %.2f, \"gbs\": %.1f}\n", name.c_str(), us, bytes / us / 1e3);
    fflush(stdout);
}

int main(int argc, char **argv)
{
    const uint32_t S = argc > 1 ? uint32_t(atoi(argv[1])) : 65536, P = 256;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    g_sms = prop.multiProcessorCount;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    const size_t region = size_t(S) * P * 8;
    char *slot, *cf, *ring, *flat;
    long long *first, *at;
    CK(cudaMalloc(&slot, region));
    CK(cudaMalloc(&cf, region));
    CK(cudaMalloc(&ring, region * kSlices));
    CK(cudaMalloc(&flat, region * 3));
    CK(cudaMalloc(&first, size_t(S) * 8));
    CK(cudaMalloc(&at, size_t(S) * 8));
    CK(cudaMemset(first, 0, size_t(S) * 8));
    CK(cudaMemset(at, 0, size_t(S) * 8));
    Regions r = {slot, cf, ring, first, at, S, P, 0x53581255ull, 1e-6f};
    auto with_slice = [&](int i) {
        Regions q = r;
        q.ring = ring + size_t(i % kSlices) * region;
        return q;
    };
    const double bytes3 = 3.0 * region;
    printf("{\"device\": \"%s\", \"sms\": %d, \"streams\": %u, \"period\": %u, \"bytes_3_regions\": %.0f}\n", prop.name, g_sms, S, P, bytes3);

    report("memset_3_regions", time_us([&](int i) {
               CK(cudaMemsetAsync(slot, i, region));
               CK(cudaMemsetAsync(cf, i, region));
               CK(cudaMemsetAsync(ring + size_t(i % kSlices) * region, i, region));
           }),
           bytes3);
    report("memset_1_contiguous", time_us([&](int i) { CK(cudaMemsetAsync(flat, i, 3 * region)); }), bytes3);
    report("memset_1_region", time_us([&](int i) { CK(cudaMemsetAsync(slot, i, region)); }), double(region));

#define RUN(NAME, KERNEL, BYTES)                                                                   \
    for (int c : ctas)                                                                             \
        report(std::string(NAME) + "_cps" + std::to_string(c),                                     \
               time_us([&](int i) { KERNEL<<<g_sms * c, 256>>>(with_slice(i)); }), BYTES);





    if (argc > 2 && atoi(argv[2]) == 5) { // fifth pass: the library's own plan and data kernels, apart and together
        BankState b = {};
        b.nstreams = S, b.period = P, b.ring = 65536 / P * P, b.sample_rate = 75000.0, b.thr2 = 0.0f, b.seed = 7;
        long long **ll[] = {&b.clock, &b.rx_position, &b.tx_position, &b.rx_time_ns, &b.rx_first_frame, &b.tx_write_position,
                            &b.tx_gap_start, &b.tx_gap_length, &b.tx_ring_offset};
        for (auto q : ll) {
            CK(cudaMalloc(q, size_t(S) * 8));
            CK(cudaMemset(*q, 0, size_t(S) * 8));
        }
        int **ii[] = {&b.rx_ret, &b.rx_flags, &b.tx_ret};
        for (auto q : ii)
            CK(cudaMalloc(q, size_t(S) * 4));
        CK(cudaMalloc(&b.rx_blocks, size_t(S) * sizeof(BlockDesc)));
        b.capture_stage = slot;
        CK(cudaFree(ring));
        CK(cudaFree(flat));
        const size_t ring_bytes = size_t(S) * b.ring * 8;
        CK(cudaMalloc(&b.playback_ring, ring_bytes));
        CK(cudaMemset(b.playback_ring, 0, ring_bytes));
        const long long lat = 10240000;
        const uint64_t vectors = uint64_t(S) * (P / 2);
        for (int blk : {32, 64, 128, 256})
            report("plan_kernel_block" + std::to_string(blk),
                   time_us([&](int) { bank_plan_repeat_kernel<<<(S + blk - 1) / blk, blk>>>(b, cf, lat); }, 100), bytes3);
        report("data_kernel_u2", time_us([&](int) { bank_repeat_data_kernel<2, IdentityHook><<<unsigned((vectors + 511) / 512), 256>>>(b, cf, false, IdentityHook()); }, 50), bytes3);
        report("data_kernel_u4", time_us([&](int) { bank_repeat_data_kernel<4, IdentityHook><<<unsigned((vectors + 1023) / 1024), 256>>>(b, cf, false, IdentityHook()); }, 50), bytes3);
        report("data_kernel_u2_external", time_us([&](int) { bank_repeat_data_kernel<2, IdentityHook><<<unsigned((vectors + 511) / 512), 256>>>(b, cf, true, IdentityHook()); }, 50), bytes3);
        report("data_kernel_u4_external", time_us([&](int) { bank_repeat_data_kernel<4, IdentityHook><<<unsigned((vectors + 1023) / 1024), 256>>>(b, cf, true, IdentityHook()); }, 50), bytes3);
        report("plan_then_data_u2_programmatic", time_us([&](int) { CK((launch_bank_planned<kBankModeRepeat, 2>(b, cf, false, SX_HAS_TIME, nullptr, lat, 0, IdentityHook()))); }, 50), bytes3);
        report("plan_then_data_u4_programmatic", time_us([&](int) { CK((launch_bank_planned<kBankModeRepeat, 4>(b, cf, false, SX_HAS_TIME, nullptr, lat, 0, IdentityHook()))); }, 50), bytes3);
        report("plan_then_data_u2_programmatic_external", time_us([&](int) { CK((launch_bank_planned<kBankModeRepeat, 2>(b, cf, true, SX_HAS_TIME, nullptr, lat, 0, IdentityHook()))); }, 50), bytes3);
        {
            cudaStream_t cs;
            CK(cudaStreamCreate(&cs));
            cudaGraph_t graph;
            cudaGraphExec_t exec;
            CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            CK((launch_bank_planned<kBankModeRepeat, 2>(b, cf, false, SX_HAS_TIME, nullptr, lat, cs, IdentityHook())));
            CK(cudaStreamEndCapture(cs, &graph));
            CK(cudaGraphInstantiate(&exec, graph, 0));
            report("plan_then_data_u2_programmatic_graph", time_us([&](int) { CK(cudaGraphLaunch(exec, 0)); }, 50), bytes3);
        }
        report("group_kernel_v100", time_us([&](int) { bank_repeat_kernel<<<740, 256>>>(b, cf, lat, false); }, 50), bytes3);
        return 0;
    }
    if (argc > 2 && atoi(argv[2]) == 4) {
        CK(cudaFree(slot));
        CK(cudaFree(cf));
        CK(cudaFree(ring));
        CK(cudaFree(flat));
        const uint64_t maxframes = uint64_t(1) << 27;
        char *a, *b, *c;
        CK(cudaMalloc(&a, maxframes * 8));
        CK(cudaMalloc(&b, maxframes * 8));
        CK(cudaMalloc(&c, maxframes * 8));
        CK(cudaMemset(a, 0x5a, maxframes * 8));
        for (int lg : {27, 24, 21, 17}) {
            const uint64_t frames = uint64_t(1) << lg, nvec = frames / 2;
            ConvArgs ca = {a, b, c, nvec, 1e-6f};
            const double bytes16 = 16.0 * frames, bytes12 = 12.0 * frames;
            const std::string tag = "_2^" + std::to_string(lg);
            const int reps = lg >= 24 ? 20 : 200;
#define RUN_C2(NAME, OP, U_, B_, W_, SH_)                                                          \
    report(std::string(NAME) + tag, time_us([&](int) { convert_np2_kernel<OP, U_, B_, W_, SH_><<<unsigned((nvec * 16 / W_ + B_ * U_ - 1) / (B_ * U_)), B_>>>(ca); }, reps), bytes16);
            RUN_C2("rx_np_u2_b256_w16_noalloc", RxCf32, 2, 256, 16, 1)
            RUN_C2("rx_np_u2_b256_w16_default", RxCf32, 2, 256, 16, 0)
            RUN_C2("rx_np_u2_b256_w16_cs", RxCf32, 2, 256, 16, 2)
            RUN_C2("rx_np_u3_b256_w16", RxCf32, 3, 256, 16, 1)
            RUN_C2("rx_np_u2_b128_w16", RxCf32, 2, 128, 16, 1)
            RUN_C2("rx_np_u4_b128_w16", RxCf32, 4, 128, 16, 1)
            RUN_C2("rx_np_u1_b512_w16", RxCf32, 1, 512, 16, 1)
            RUN_C2("rx_np_u2_b512_w16", RxCf32, 2, 512, 16, 1)
            RUN_C2("rx_np_u1_b1024_w16", RxCf32, 1, 1024, 16, 1)
            RUN_C2("rx_np_u1_b256_w32_evict_first", RxCf32, 1, 256, 32, 1)
            RUN_C2("rx_np_u2_b256_w32_evict_first", RxCf32, 2, 256, 32, 1)
            RUN_C2("rx_np_u1_b256_w32_plain_store", RxCf32, 1, 256, 32, 0)
            RUN_C2("rx_np_u1_b128_w32_evict_first", RxCf32, 1, 128, 32, 1)
            RUN_C2("tx_np_u2_b256_w16_noalloc", TxCf32, 2, 256, 16, 1)
            RUN_C2("tx_np_u1_b256_w32_evict_first", TxCf32, 1, 256, 32, 1)
            RUN_C2("tx_np_u2_b128_w16", TxCf32, 2, 128, 16, 1)
#define RUN_N(NAME, OP, U_, B_)                                                                    \
    report(std::string(NAME) + tag, time_us([&](int) { convert_np_narrow_kernel<OP, U_, B_><<<unsigned((nvec / 2 + B_ * U_ - 1) / (B_ * U_)), B_>>>(ca); }, reps), bytes12);
            RUN_N("rx_cs16_np_u1_b256", RxCs16, 1, 256)
            RUN_N("rx_cs16_np_u2_b256", RxCs16, 2, 256)
            RUN_N("rx_cs16_np_u2_b128", RxCs16, 2, 128)
            RUN_N("tx_cs16_np_u1_b256", TxCs16, 1, 256)
            RUN_N("tx_cs16_np_u2_b256", TxCs16, 2, 256)
            RUN_N("tx_cs16_np_u2_b128", TxCs16, 2, 128)
        }
        return 0;
    }
    if (argc > 2 && atoi(argv[2]) == 3) { // third pass: converters on hardware-scheduled CTAs; the bank with its plan
        {
            PlanArrays p;
            long long **ll[] = {&p.clock, &p.rx_pos, &p.tx_pos, &p.rx_time, &p.first, &p.at, &p.gap, &p.start};
            for (auto q : ll) {
                CK(cudaMalloc(q, size_t(S) * 8));
                CK(cudaMemset(*q, 0, size_t(S) * 8));
            }
            int **ii[] = {&p.rx_ret, &p.rx_flags, &p.tx_ret};
            for (auto q : ii)
                CK(cudaMalloc(q, size_t(S) * 4));
            p.rate = 75000.0;
            const uint64_t total = uint64_t(S) * P / 2;
#define RUN_BANK(NAME, U_, B_, EXT_, BYTES)                                                        \
    report(NAME, time_us([&](int i) { bank_np_kernel<U_, B_, EXT_><<<unsigned((total + B_ * U_ - 1) / (B_ * U_)), B_>>>(with_slice(i), p); }), BYTES);
            RUN_BANK("bank_np_u1_b256", 1, 256, false, bytes3)
            RUN_BANK("bank_np_u2_b256", 2, 256, false, bytes3)
            RUN_BANK("bank_np_u4_b256", 4, 256, false, bytes3)
            RUN_BANK("bank_np_u8_b256", 8, 256, false, bytes3)
            RUN_BANK("bank_np_u2_b128", 2, 128, false, bytes3)
            RUN_BANK("bank_np_u4_b128", 4, 128, false, bytes3)
            RUN_BANK("bank_np_u2_b512", 2, 512, false, bytes3)
            RUN_BANK("bank_np_u4_b512", 4, 512, false, bytes3)
            RUN_BANK("bank_np_u2_b1024", 2, 1024, false, bytes3)
            RUN_BANK("bank_np_external_u2_b256", 2, 256, true, bytes3)
            RUN_BANK("bank_np_external_u4_b256", 4, 256, true, bytes3)
            RUN_BANK("bank_np_external_u8_b256", 8, 256, true, bytes3)
            RUN_BANK("bank_np_external_u4_b512", 4, 512, true, bytes3)
        }
        CK(cudaFree(slot));
        CK(cudaFree(cf));
        CK(cudaFree(ring));
        CK(cudaFree(flat));
        const uint64_t frames = uint64_t(1) << 27, nvec = frames / 2;
        char *a, *b, *c;
        CK(cudaMalloc(&a, frames * 8));
        CK(cudaMalloc(&b, frames * 8));
        CK(cudaMalloc(&c, frames * 8));
        CK(cudaMemset(a, 0x5a, frames * 8));
        ConvArgs ca = {a, b, c, nvec, 1e-6f};
        const double bytes16 = 16.0 * frames, bytes24 = 24.0 * frames;
        report("memcpy_d2d_1GiB", time_us([&](int) { CK(cudaMemcpyAsync(b, a, frames * 8, cudaMemcpyDeviceToDevice)); }, 20), bytes16);
#define RUN_CONV(NAME, KERNEL, U_, BYTES)                                                          \
    report(NAME, time_us([&](int) { KERNEL<<<unsigned((nvec + 256 * U_ - 1) / (256 * U_)), 256>>>(ca); }, 20), BYTES);
        RUN_CONV("rx_np_u1", (convert_np_kernel<RxCf32, 1, 0>), 1, bytes16)
        RUN_CONV("rx_np_u2", (convert_np_kernel<RxCf32, 2, 0>), 2, bytes16)
        RUN_CONV("rx_np_u4", (convert_np_kernel<RxCf32, 4, 0>), 4, bytes16)
        RUN_CONV("rx_np_u8", (convert_np_kernel<RxCf32, 8, 0>), 8, bytes16)
        RUN_CONV("rx_np_u16", (convert_np_kernel<RxCf32, 16, 0>), 16, bytes16)
        RUN_CONV("rx_np_nc_u4", (convert_np_kernel<RxCf32, 4, 1>), 4, bytes16)
        RUN_CONV("rx_np_nc_u8", (convert_np_kernel<RxCf32, 8, 1>), 8, bytes16)
        RUN_CONV("rx_np_adjacent_u2", (convert_np_adjacent_kernel<RxCf32, 2>), 2, bytes16)
        RUN_CONV("rx_np_adjacent_u4", (convert_np_adjacent_kernel<RxCf32, 4>), 4, bytes16)
        RUN_CONV("tx_np_u2", (convert_np_kernel<TxCf32, 2, 0>), 2, bytes16)
        RUN_CONV("tx_np_u4", (convert_np_kernel<TxCf32, 4, 0>), 4, bytes16)
        RUN_CONV("tx_np_u8", (convert_np_kernel<TxCf32, 8, 0>), 8, bytes16)
        RUN_CONV("loopback_np_u2", (loopback_np_kernel<2>), 2, bytes24)
        RUN_CONV("loopback_np_u4", (loopback_np_kernel<4>), 4, bytes24)
        RUN_CONV("loopback_np_u8", (loopback_np_kernel<8>), 8, bytes24)
        return 0;
    }
    if (argc > 2) { // second pass: the flat pattern and CTA-contiguous chunks
        const uint64_t total = uint64_t(S) * P / 2;
        {
            const int ctas[] = {4, 8};
            RUN("store_flat_noalloc_u2_r3", (store_flat_kernel<1, 2>), bytes3)
            RUN("store_flat_noalloc_u4_r3", (store_flat_kernel<1, 4>), bytes3)
            RUN("store_flat_noalloc_u8_r3", (store_flat_kernel<1, 8>), bytes3)
            RUN("store_flat_noalloc_u16_r3", (store_flat_kernel<1, 16>), bytes3)
            RUN("store_chunk_persistent_u4", (store_chunk_kernel<1, 4, true>), bytes3)
            RUN("store_chunk_persistent_u8", (store_chunk_kernel<1, 8, true>), bytes3)
            RUN("store_chunk_persistent_u16", (store_chunk_kernel<1, 16, true>), bytes3)
            RUN("fused_grid_flat_u4", (fused_grid_flat_kernel<1, 4, 1>), bytes3)
            RUN("fused_grid_flat_u2", (fused_grid_flat_kernel<1, 2, 1>), bytes3)
            RUN("fused_grid_flat_u8", (fused_grid_flat_kernel<1, 8, 1>), bytes3)
            RUN("fused_chunk_persistent_u4", (fused_chunk_kernel<1, 4, 1, true>), bytes3)
            RUN("fused_chunk_persistent_u8", (fused_chunk_kernel<1, 8, 1, true>), bytes3)
        }
#define RUN_NP(NAME, KERNEL, U_)                                                                   \
    report(NAME, time_us([&](int i) { KERNEL<<<unsigned((total + 256 * U_ - 1) / (256 * U_)), 256>>>(with_slice(i)); }), bytes3);
        RUN_NP("store_chunk_np_u1", (store_chunk_kernel<1, 1, false>), 1)
        RUN_NP("store_chunk_np_u2", (store_chunk_kernel<1, 2, false>), 2)
        RUN_NP("store_chunk_np_u4", (store_chunk_kernel<1, 4, false>), 4)
        RUN_NP("store_chunk_np_u8", (store_chunk_kernel<1, 8, false>), 8)
        RUN_NP("store_chunk_np_u16", (store_chunk_kernel<1, 16, false>), 16)
        RUN_NP("store_chunk_np_default_u4", (store_chunk_kernel<0, 4, false>), 4)
        RUN_NP("store_flat_np_u2", (store_flat_np_kernel<1, 2>), 2)
        RUN_NP("store_flat_np_u4", (store_flat_np_kernel<1, 4>), 4)
        RUN_NP("store_flat_np_u8", (store_flat_np_kernel<1, 8>), 8)
        RUN_NP("fused_chunk_np_u2", (fused_chunk_kernel<1, 2, 1, false>), 2)
        RUN_NP("fused_chunk_np_u4", (fused_chunk_kernel<1, 4, 1, false>), 4)
        RUN_NP("fused_chunk_np_u8", (fused_chunk_kernel<1, 8, 1, false>), 8)
        // repeatability of the first pass's outliers
        {
            const int ctas[] = {8};
            RUN("again_store_only_noalloc_u4_r3", (store_only_kernel<1, 4, 3>), bytes3)
            RUN("again_store_flat_noalloc_u4_r3", (store_flat_kernel<1, 4>), bytes3)
            RUN("again_fused_flat_noalloc_u4", (fused_flat_kernel<1, 4, 1, false>), bytes3)
        }
        report("again_memset_1_contiguous", time_us([&](int i) { CK(cudaMemsetAsync(flat, i, 3 * region)); }), bytes3);
        return 0;
    }
    {
        const int ctas[] = {2, 4, 8};
        RUN("store_only_default_u4_r3", (store_only_kernel<0, 4, 3>), bytes3)
        RUN("store_only_noalloc_u4_r3", (store_only_kernel<1, 4, 3>), bytes3)
        RUN("store_only_cs_u4_r3", (store_only_kernel<2, 4, 3>), bytes3)
        RUN("store_only_cg_u4_r3", (store_only_kernel<3, 4, 3>), bytes3)
        RUN("store_only_noalloc_u1_r3", (store_only_kernel<1, 1, 3>), bytes3)
        RUN("store_only_noalloc_u2_r3", (store_only_kernel<1, 2, 3>), bytes3)
        RUN("store_only_noalloc_u4_r1", (store_only_kernel<1, 4, 1>), bytes3 / 3)
        RUN("store_only_noalloc_u4_r2", (store_only_kernel<1, 4, 2>), bytes3 * 2 / 3)
        RUN("store_only_256bit_u2_r3", (store_only256_kernel<2>), bytes3)
        RUN("store_only_256bit_u1_r3", (store_only256_kernel<1>), bytes3)
        RUN("store_flat_noalloc_u4_r3", (store_flat_kernel<1, 4>), bytes3)
        RUN("store_flat_noalloc_u1_r3", (store_flat_kernel<1, 1>), bytes3)
        RUN("store_flat_default_u4_r3", (store_flat_kernel<0, 4>), bytes3)
    }
    {
        const int ctas[] = {2, 4, 6, 8};
        RUN("compute_only_u4", (compute_only_kernel<4>), bytes3)
        RUN("compute_only_u1", (compute_only_kernel<1>), bytes3)
    }
    {
        const int ctas[] = {2, 3, 4, 6, 8};
        RUN("fused_flat_noalloc_u4", (fused_flat_kernel<1, 4, 1, false>), bytes3)
        RUN("fused_flat_noalloc_u2", (fused_flat_kernel<1, 2, 1, false>), bytes3)
        RUN("fused_flat_noalloc_u1", (fused_flat_kernel<1, 1, 1, false>), bytes3)
        RUN("fused_flat_default_u2", (fused_flat_kernel<0, 2, 1, false>), bytes3)
        RUN("fused_flat_cs_u2", (fused_flat_kernel<2, 2, 1, false>), bytes3)
        RUN("fused_flat_256bit_u1", (fused_flat_kernel<1, 1, 1, true>), bytes3)
        RUN("fused_flat_256bit_u2", (fused_flat_kernel<1, 2, 1, true>), bytes3)
    }
    return 0;
}
