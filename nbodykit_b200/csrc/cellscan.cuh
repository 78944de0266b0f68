// Exclusive scan of per-cell counts into cell starts, shared by the counting sorts of fof.cu and paircount.cu.
// Three launches: segment totals, one CTA scanning the totals, then every segment scans itself from its carry.
#pragma once
#include "common.cuh"

#define NBK_SCAN_SEG 4096       // elements per CTA of the offset scan (1024 threads x 4)

// segments of the scan of C counts (the scratch `segtot` holds this many + 1 ints)
static inline int64_t nbk_scan_nseg(int64_t C) { return (C + 1 + NBK_SCAN_SEG - 1) / NBK_SCAN_SEG; }

static __global__ void __launch_bounds__(1024) k_scan_seg_totals(const int *__restrict__ cnt, int64_t C, int *__restrict__ segtot) {
    __shared__ int wt[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * NBK_SCAN_SEG + threadIdx.x * 4;
    int s = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) if (i + j < C) s += cnt[i + j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) wt[wid] = s;
    __syncthreads();
    if (wid == 0) {
        int x = wt[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) segtot[blockIdx.x] = x;
    }
}

static __device__ __forceinline__ int block_excl_scan(int v, int *wt, int *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int nn = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += nn;
    }
    if (lane == 31) wt[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int x = wt[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int nn = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += nn;
        }
        wt[lane] = x;
    }
    __syncthreads();
    int r = (wid ? wt[wid - 1] : 0) + inc - v;
    *total = wt[31];
    __syncthreads();
    return r;
}

static __global__ void __launch_bounds__(1024) k_scan_totals(int *__restrict__ segtot, int nseg) {
    __shared__ int wt[32];
    int carry = 0;
    for (int base = 0; base < nseg; base += 1024) {
        int i = base + threadIdx.x;
        int v = i < nseg ? segtot[i] : 0, tot;
        int e = block_excl_scan(v, wt, &tot);
        if (i < nseg) segtot[i] = carry + e;
        carry += tot;
    }
}

static __global__ void __launch_bounds__(1024)
k_scan_seg(const int *__restrict__ cnt, int64_t C, const int *__restrict__ segtot, int *__restrict__ cstart, int n) {
    __shared__ int wt[32];
    const int64_t i = (int64_t)blockIdx.x * NBK_SCAN_SEG + threadIdx.x * 4;
    int v[4];
#pragma unroll
    for (int j = 0; j < 4; j++) v[j] = (i + j < C) ? cnt[i + j] : 0;
    int tot;
    int run = segtot[blockIdx.x] + block_excl_scan(v[0] + v[1] + v[2] + v[3], wt, &tot);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (i + j < C) cstart[i + j] = run;
        run += v[j];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) cstart[C] = n;
}

// cstart[0..C] = exclusive scan of cnt[0..C), cstart[C] = n (the sum of the counts)
static inline int nbk_cell_scan(const int *cnt, int64_t C, int *segtot, int *cstart, int n, cudaStream_t s) {
    const int nseg = (int)nbk_scan_nseg(C);
    k_scan_seg_totals<<<nseg, 1024, 0, s>>>(cnt, C, segtot);
    NBK_LAUNCHED();
    k_scan_totals<<<1, 1024, 0, s>>>(segtot, nseg);
    NBK_LAUNCHED();
    k_scan_seg<<<nseg, 1024, 0, s>>>(cnt, C, segtot, cstart, n);
    NBK_LAUNCHED();
    return NBK_OK;
}
