// select.cuh -- order statistics of a column of doubles in global memory, by one thread block: the order-preserving
// 64-bit key of a double and an 8-bit radix select on it.  Used by posterior.cu (percentiles of long PSD columns) and
// survey.cu (the Pareto-tail cut of carma_multi_laplace).
#pragma once

namespace carma {

__device__ __forceinline__ unsigned long long order_key(double v) {   // a < b  <=>  key(a) < key(b) (non-NaN)
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

struct SelectSmem {
    unsigned hist[256];
    unsigned long long bcast[2], cnt_le, min_gt;
};

// Order statistics k and min(k + 1, n - 1) (0-based), as order keys, of a column x of n doubles in global memory: eight
// passes of an 8-bit radix select for k, then one pass for k + 1 (ka again if it occurs more than k + 1 times, else the
// smallest larger key).  Whole block.
inline __device__ void block_select_pair(const double* __restrict__ x, size_t n, size_t k, SelectSmem& sm,
                                  unsigned long long* ka_out, unsigned long long* kb_out) {
    unsigned long long prefix = 0, mask = 0;
    size_t kk = k;
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) sm.hist[i] = 0;
        __syncthreads();
        for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned long long v = order_key(x[i]);
            if ((v & mask) == prefix) atomicAdd(&sm.hist[(v >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            size_t acc = 0;
            int dsel = 255;
            for (int dg = 0; dg < 256; dg++) {
                if (acc + sm.hist[dg] > kk) { dsel = dg; break; }
                acc += sm.hist[dg];
            }
            sm.bcast[0] = (unsigned long long)dsel;
            sm.bcast[1] = kk - acc;
        }
        __syncthreads();
        prefix |= sm.bcast[0] << shift;
        mask |= 255ull << shift;
        kk = (size_t)sm.bcast[1];
        __syncthreads();
    }
    unsigned long long kb = prefix;
    if (k + 1 < n) {
        if (threadIdx.x == 0) { sm.cnt_le = 0; sm.min_gt = ~0ull; }
        __syncthreads();
        unsigned long long my_cnt = 0, my_min = ~0ull;
        for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
            const unsigned long long v = order_key(x[i]);
            if (v <= prefix) my_cnt++;
            else my_min = my_min < v ? my_min : v;
        }
        atomicAdd(&sm.cnt_le, my_cnt);
        atomicMin(&sm.min_gt, my_min);
        __syncthreads();
        if (sm.cnt_le <= k + 1) kb = sm.min_gt;
        __syncthreads();
    }
    *ka_out = prefix;
    *kb_out = kb;
}

}  // namespace carma
