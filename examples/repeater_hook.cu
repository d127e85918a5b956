// repeater_hook.cu -- the reference repeater's DSP, compiled INTO the fused bank iteration
// through include/sx_hook.cuh.
//
// example/linear_repeater.py:100-106 (between its two channel filters):
//         s *= 1000.0
//         clip_signal(s)          # s /= np.maximum(np.abs(s), 1.0)        (:87-89)
//         s *= 0.3
// is the functor below.  The scipy IIR channel filters around it carry state from block to block;
// they are the library's sxgpu_iir cascades, which sx_example_repeat_filtered_clip_gain runs before
// and after the functor in the same launch: the script's whole process().
//
// Arithmetic, chosen so that a CPU restatement can match it bit for bit (tests/test_gpu_hook.py):
// every step is one correctly rounded IEEE operation, nothing is contracted; |s| is
// float(sqrt(double(re)^2 + double(im)^2)); the division is a multiplication by 1.0f / max(|s|, 1)
// as in numpy's complex-by-real division.  numpy's own np.abs is a few ulp less exact than that,
// so the literal numpy expression agrees to within a stated tolerance, not bit for bit.
#include "../include/sx_hook.cuh"

struct ClipGain {
    float pre, post;
    __device__ __forceinline__ void operator()(sx::Pack<4> &v, uint64_t, uint32_t) const
    {
#pragma unroll
        for (int k = 0; k < 2; k++) {
            float re = __fmul_rn(__uint_as_float(v.w[2 * k]), pre);
            float im = __fmul_rn(__uint_as_float(v.w[2 * k + 1]), pre);
            const double m2 = __dadd_rn(__dmul_rn(double(re), double(re)), __dmul_rn(double(im), double(im)));
            const float mag = __double2float_rn(__dsqrt_rn(m2));
            const float scale = __fdiv_rn(1.0f, fmaxf(mag, 1.0f));
            re = __fmul_rn(__fmul_rn(re, scale), post);
            im = __fmul_rn(__fmul_rn(im, scale), post);
            v.w[2 * k] = __float_as_uint(re);
            v.w[2 * k + 1] = __float_as_uint(im);
        }
    }
};

// The same stage as a kernel of its own, for the two-launch form
// (sxgpu_bank_repeat_begin -> this -> sxgpu_bank_repeat_end).
__global__ void clip_gain_kernel(float *cf32, uint64_t nvec, ClipGain op)
{
    for (uint64_t v = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; v < nvec; v += uint64_t(gridDim.x) * blockDim.x) {
        uint4 q = reinterpret_cast<uint4 *>(cf32)[v];
        sx::Pack<4> p;
        p.w[0] = q.x, p.w[1] = q.y, p.w[2] = q.z, p.w[3] = q.w;
        op(p, 0, 0);
        reinterpret_cast<uint4 *>(cf32)[v] = make_uint4(p.w[0], p.w[1], p.w[2], p.w[3]);
    }
}

extern "C" {

// One repeater iteration of every stream of the bank with the clipper inside the fused kernel.
int sx_example_repeat_clip_gain(sxgpu_bank *bank, void *d_cf32, long long rx_time_offset_ns, float pre_gain,
                                float post_gain, void *stream)
{
    return sx::bank_repeat_with(bank, d_cf32, rx_time_offset_ns, static_cast<cudaStream_t>(stream),
                                ClipGain{pre_gain, post_gain});
}

// The script's whole process() inside the fused iteration: `pre` filter, the clipper, `post` filter.
int sx_example_repeat_filtered_clip_gain(sxgpu_bank *bank, sxgpu_iir *pre, sxgpu_iir *post, void *d_cf32,
                                         long long rx_time_offset_ns, float pre_gain, float post_gain, void *stream)
{
    return sx::bank_repeat_with(bank, d_cf32, rx_time_offset_ns, static_cast<cudaStream_t>(stream),
                                ClipGain{pre_gain, post_gain}, pre, post);
}

// The same iteration as three launches around an ordinary kernel, the CF32 block kept in L2.
int sx_example_repeat_clip_gain_split(sxgpu_bank *bank, void *d_cf32, uint64_t nframes_total,
                                      long long rx_time_offset_ns, float pre_gain, float post_gain, void *stream)
{
    int rc = sxgpu_bank_repeat_begin(bank, d_cf32, stream);
    if (rc != SXGPU_OK)
        return rc;
    const uint64_t nvec = nframes_total / 2;
    const unsigned grid = unsigned(nvec / 256 + 1 < 148 * 8 ? nvec / 256 + 1 : 148 * 8);
    clip_gain_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<float *>(d_cf32), nvec,
                                                                         ClipGain{pre_gain, post_gain});
    if (cudaGetLastError() != cudaSuccess)
        return SXGPU_ERR_CUDA;
    return sxgpu_bank_repeat_end(bank, d_cf32, rx_time_offset_ns, stream);
}

} // extern "C"
