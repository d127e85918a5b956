// sx_hook.cuh -- user DSP between the RX and the TX conversion, INSIDE the fused bank iteration.
//
// The reference's repeater is read -> process(buf) -> timed write
// (example/linear_repeater.py:50-71; the DSP at :78-109).  sxgpu_bank_repeat() is that loop for
// thousands of streams in one launch with an identity process().  This header lets an
// application compile its own process() into the same kernel: the CF32 samples are handed to a
// device functor while they are still in registers, between RxCf32 and TxCf32, so the user stage
// costs no extra pass over memory.  Header-only; include it from a .cu file built for sm_100a
// and link against libsxgpu.so:
//
//     struct Gain { float g;
//         __device__ void operator()(sx::Pack<4> &v, uint64_t stream, uint32_t frame) const {
//             for (int k = 0; k < 4; k++) v.w[k] = __float_as_uint(__uint_as_float(v.w[k]) * g); } };
//     sx::bank_repeat_with(bank, d_cf32, offset_ns, cuda_stream, Gain{0.5f});
//
// The functor sees two consecutive complex samples of one stream per call --
// v.w = {re0, im0, re1, im1} as float bits, `frame` = index of the first within the block -- and
// may change them in place; what it leaves is what lands in the caller's CF32 block and what
// the TX conversion packs.  Calls for one block are spread over the lanes of a warp in no
// particular order, so the functor must be memoryless across samples (gain, clipper, mixer with
// a per-frame phase, ...).  Filters with state along the stream -- the channel filters of the
// reference's example -- are the library's own: the seven-argument overload below runs a
// sxgpu_iir cascade before the functor and another after it, in the same launch
//
//     sx::bank_repeat_with(bank, d_cf32, offset_ns, cuda_stream, Gain{0.5f}, pre, post);
//
// (examples/repeater_hook.cu does the script's whole process() so: filter, clip, filter).
//
// For DSP that is neither: sxgpu_bank_repeat_begin() / sxgpu_bank_repeat_end() (include/sxgpu.h)
// split the iteration around any kernel of the caller's on the same stream and keep the CF32 block
// resident in L2 in between.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "sxgpu.h"
#include "../sxxcvr_b200/csrc/sx_bank.cuh"

namespace sx {

// sxgpu_bank_repeat(bank, d_cf32, rx_time_offset_ns, stream) with `hook` applied to every pair
// of CF32 samples between the two conversions.  Same state, results and playback rings as
// sxgpu_bank_read + (hook over the CF32 block) + sxgpu_bank_write(HAS_TIME, rx time + offset).
// Needs an even period and a 16-byte aligned CF32 buffer.  Asynchronous on `stream` (which must
// be a real stream handle or the legacy default stream).
template <class Hook>
inline int bank_repeat_with(sxgpu_bank *bank, void *d_cf32, long long rx_time_offset_ns, cudaStream_t stream,
                            const Hook &hook)
{
    BankState view;
    int external = 0;
    const int rc = sxgpu_bank_device_view(bank, &view, sizeof view, &external);
    if (rc != SXGPU_OK)
        return rc;
    if (!d_cf32 || reinterpret_cast<uintptr_t>(d_cf32) % 16 || view.period % 2)
        return SXGPU_ERR_INVALID;
    int device = 0, sms = 0;
    if (cudaGetDevice(&device) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess)
        return SXGPU_ERR_CUDA;
    // Same schedule choice as the library's own fused iteration: K streams per warp round.
    auto launch = [&](auto kernel, uint64_t k) -> int {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1)
            per_sm = 1;
        const uint64_t chunks = (uint64_t(view.nstreams) + k - 1) / k;
        const uint64_t want = (chunks + 7) / 8;
        const uint64_t cap = uint64_t(sms) * uint64_t(per_sm);
        const unsigned grid = unsigned(want < cap ? (want ? want : 1) : cap);
        kernel<<<grid, 256, 0, stream>>>(view, static_cast<char *>(d_cf32), rx_time_offset_ns, external != 0, hook);
        return cudaGetLastError() == cudaSuccess ? SXGPU_OK : SXGPU_ERR_CUDA;
    };
    if (bank_is_large(view)) // the library's own choice for large banks: decisions first, then the samples
        return launch_bank_repeat_planned<2>(view, static_cast<char *>(d_cf32), rx_time_offset_ns, external != 0, stream, hook) ==
                       cudaSuccess
                   ? SXGPU_OK
                   : SXGPU_ERR_CUDA;
    if (view.nstreams <= 2048)
        return launch(bank_repeat_reg_kernel<1, Hook>, 1);
    if (view.nstreams <= 16384)
        return launch(bank_repeat_reg_kernel<2, Hook>, 2);
    return launch(bank_repeat_reg_kernel<4, Hook>, 4);
}

// The same iteration with the reference's channel filters around the functor: read -> `pre`
// cascade -> hook -> `post` cascade -> CF32 block and timed write, in one launch after the
// decisions.  Same state, results, CF32 block and playback ring as sxgpu_bank_read, then
// sxgpu_iir_apply(pre), the hook over the block, sxgpu_iir_apply(post), then sxgpu_bank_write
// (HAS_TIME, rx time + offset).  Either filter may be NULL (both: the overload above).
// With IdentityHook this is sxgpu_bank_repeat_filtered.  Needs an even period, a 16-byte aligned
// CF32 buffer and two different filters of the bank's stream count.
template <class Hook>
inline int bank_repeat_with(sxgpu_bank *bank, void *d_cf32, long long rx_time_offset_ns, cudaStream_t stream,
                            const Hook &hook, sxgpu_iir *pre, sxgpu_iir *post)
{
    BankState view;
    int external = 0;
    int rc = sxgpu_bank_device_view(bank, &view, sizeof view, &external);
    if (rc != SXGPU_OK)
        return rc;
    IirView vpre = {}, vpost = {};
    if (pre && (rc = sxgpu_iir_device_view(pre, &vpre, sizeof vpre)) != SXGPU_OK)
        return rc;
    if (post && (rc = sxgpu_iir_device_view(post, &vpost, sizeof vpost)) != SXGPU_OK)
        return rc;
    if ((pre && pre == post) || bank_repeat_iir_invalid(view, d_cf32, vpre, vpost))
        return SXGPU_ERR_INVALID;
    if (!pre && !post)
        return bank_repeat_with(bank, d_cf32, rx_time_offset_ns, stream, hook);
    return launch_bank_repeat_iir(view, static_cast<char *>(d_cf32), rx_time_offset_ns, external != 0, vpre, vpost, stream,
                                  hook) == cudaSuccess
               ? SXGPU_OK
               : SXGPU_ERR_CUDA;
}

} // namespace sx
