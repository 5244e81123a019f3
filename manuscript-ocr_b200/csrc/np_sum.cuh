// numpy's pairwise float32 summation (np.add.reduce over a contiguous vector), as a one-thread device function and as
// a CTA-wide one.  Included inside the anonymous namespace of boxes.cu (east_finish_kernel: the area-anomaly filter's
// mean and standard deviation) and of np_sum_test.cu (ms_test_np_sum_host), so both compile the same code.
#pragma once

// numpy's sum of one block of at most 128 values: 8 accumulators, then the remainder
__device__ __forceinline__ float np_block_f32(const float *a, int n)
{
    if (n < 8) {
        float r = -0.0f;
        for (int i = 0; i < n; i++) r += a[i];
        return r;
    }
    float r[8];
    for (int k = 0; k < 8; k++) r[k] = a[k];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
        for (int k = 0; k < 8; k++) r[k] += a[i + k];
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; i++) res += a[i];
    return res;
}

// numpy pairwise summation of a contiguous f32 vector (np.add.reduce; oracle.c np_pairwise_f32): a block sum for
// n <= 128, else sum(first n2) + sum(rest) with n2 = n / 2 rounded down to a multiple of 8.  The tree is walked with an
// explicit stack instead of recursion: a 120-byte frame per halving ran off the 1 KB default device stack on long
// vectors (13 frames for 300 000 values), which includes every vector that takes the one-thread path of
// np_pairwise_f32_cta (more than kPwLeafCap leaves, i.e. more than 65 536 values).
__device__ float np_pairwise_f32(const float *a, int n)
{
    constexpr int kDepth = 24;  // halvings from n < 2^31 down to 128
    int r_off[kDepth], r_len[kDepth], l_done[kDepth];  // per level: the right half, and whether its left sum is known
    float l_sum[kDepth];
    int sp = 0, off = 0, len = n;
    for (;;) {
        while (len > 128) {
            int n2 = len / 2;
            n2 -= n2 % 8;
            r_off[sp] = off + n2;
            r_len[sp] = len - n2;
            l_done[sp] = 0;
            sp++;
            len = n2;
        }
        float acc = np_block_f32(a + off, len);
        while (sp > 0 && l_done[sp - 1]) {  // a right half is complete: left + right, one level up
            sp--;
            acc = l_sum[sp] + acc;
        }
        if (sp == 0) return acc;
        l_sum[sp - 1] = acc;  // a left half is complete: the right half is next
        l_done[sp - 1] = 1;
        off = r_off[sp - 1];
        len = r_len[sp - 1];
    }
}

// The same sum by a whole CTA, bit for bit: numpy's recursion splits the vector into leaves of at most 128 elements
// and adds the leaf sums pairwise in a fixed tree.  Thread 0 lists the leaves (the split rule only), every leaf is
// summed by its own thread with the 8-accumulator loop above, thread 0 adds the leaf sums in the recursion's order.
// One thread summing 2000 areas twice out of global memory was half of east_finish_kernel's time.
constexpr int kPwLeafCap = 1024;

__device__ void pw_leaves(int off, int n, int *loff, int *llen, int &cnt)
{
    if (n <= 128) {
        if (cnt < kPwLeafCap) {
            loff[cnt] = off;
            llen[cnt] = n;
        }
        cnt++;
    } else {
        int n2 = n / 2;
        n2 -= n2 % 8;
        pw_leaves(off, n2, loff, llen, cnt);
        pw_leaves(off + n2, n - n2, loff, llen, cnt);
    }
}

__device__ float pw_combine(int n, const float *lsum, int &cnt)
{
    if (n <= 128) return lsum[cnt++];
    int n2 = n / 2;
    n2 -= n2 % 8;
    const float lo = pw_combine(n2, lsum, cnt);
    const float hi = pw_combine(n - n2, lsum, cnt);
    return lo + hi;
}

// called by every thread of the CTA; s_loff / s_llen / s_lsum hold kPwLeafCap entries each
__device__ float np_pairwise_f32_cta(const float *a, int n, int *s_loff, int *s_llen, float *s_lsum, int *s_cnt,
                                     float *s_out)
{
    if (threadIdx.x == 0) {
        int c = 0;
        pw_leaves(0, n, s_loff, s_llen, c);
        *s_cnt = c;
    }
    __syncthreads();
    const int c = *s_cnt;
    if (c > kPwLeafCap) {
        if (threadIdx.x == 0) *s_out = np_pairwise_f32(a, n);
    } else {
        for (int t = threadIdx.x; t < c; t += blockDim.x) s_lsum[t] = np_pairwise_f32(a + s_loff[t], s_llen[t]);
        __syncthreads();
        if (threadIdx.x == 0) {
            int k = 0;
            *s_out = pw_combine(n, s_lsum, k);
        }
    }
    __syncthreads();
    const float r = *s_out;
    __syncthreads();  // s_out and the leaf tables may be reused by the next call
    return r;
}
