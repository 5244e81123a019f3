// Test-only (ms_test_np_sum_host): numpy's pairwise float32 sums of np_sum.cuh, evaluated on the device as
// east_finish_kernel evaluates them for the area-anomaly filter -- a CTA of its 1024 threads with leaf tables of its
// sizes in shared memory.  A translation unit of its own: a second caller inside boxes.cu would change how the compiler
// inlines and allocates registers for these functions in east_finish_kernel.
#include "ms_internal.cuh"

namespace {

#include "np_sum.cuh"

// one CTA per vector: out_cta = np_pairwise_f32_cta (leaf-parallel, one thread beyond kPwLeafCap leaves),
// out_serial = np_pairwise_f32 on one thread
__global__ void __launch_bounds__(1024) np_sum_test_kernel(const float *__restrict__ values,
                                                          const int64_t *__restrict__ offsets,
                                                          const int32_t *__restrict__ lengths,
                                                          float *__restrict__ out_serial, float *__restrict__ out_cta)
{
    ms_pdl_wait();
    const int v = blockIdx.x;
    const float *a = values + offsets[v];
    const int n = lengths[v];
    __shared__ int s_loff[kPwLeafCap], s_llen[kPwLeafCap], s_pwcnt;
    __shared__ float s_lsum[kPwLeafCap], s_pwout;
    const float cta = np_pairwise_f32_cta(a, n, s_loff, s_llen, s_lsum, &s_pwcnt, &s_pwout);
    if (threadIdx.x == 0) {
        out_cta[v] = cta;
        out_serial[v] = np_pairwise_f32(a, n);
    }
}

}  // namespace

int msk_test_np_sum(ms_ctx *ctx, const float *values, const int64_t *offsets, const int32_t *lengths, int n_vec,
                    float *out_serial, float *out_cta, cudaStream_t st)
{
    if (n_vec <= 0) return MS_OK;
    ms_launch(np_sum_test_kernel, n_vec, 1024, 0, st, values, offsets, lengths, out_serial, out_cta);
    MS_LAUNCH_CHECK(ctx);
    return MS_OK;
}
