// cuFFT-free 3-D real<->complex FFT (RealField.r2c / ComplexField.c2r: base/mesh.py:228,237;
// source/mesh/catalog.py:341-351).  Forward is normalised by 1/prod(N), backward is not
// (source/mesh/array.py:36-37, fftpower.py:126-128).
//
// Structure: three line passes, each one read + one write of the field (HBM-bound):
//   z pass  : rows are contiguous; real row of Nz -> packed complex FFT of Nz/2 -> Nz/2+1 modes
//   y pass  : lines strided by Nzc, tiles of B adjacent kz columns  (B * sizeof(cplx) = 128-byte runs)
//   x pass  : lines strided by Ny*Nzc, tiles of B adjacent (y,kz) elements
// Default kernels (round 2), built around the copy engine so that the warps only run butterflies:
//   k_fft_lines_tma   lines of 256 / 512 / 1024: row groups stream through a ring of shared-memory slots as 4-D tensor-map
//                     boxes (cp.async.bulk.tensor + mbarrier), one 64-point FFT per warp, one radix-R combine per tile
//   k_fft_z_r2c_tma   rows of 256 / 512 / 1024 reals: warp-per-row, private ring of row buffers filled by 1-D bulk copies
// Older families, still serving short lines, c8 lines whose rows are not 16-byte aligned, the backward z pass and the
// NBK_FFT_LINES=rg|smem knob: the register-I/O kernels (k_fft_lines_rg, k_fft_z_r2c_rg: first radix-8 stage straight from
// global memory, last stage straight to the digit-reversed frequency rows, [N][B+1] padded tiles in between) and the
// shared-memory kernels (k_fft_lines with cp.async double buffering, k_fft_z_r2c, k_fft_z_c2r).
// Decimation-in-frequency radix-8 butterflies in registers throughout (+ one radix-4 / radix-2 stage for the remainder of
// log2 N).  Twiddles: f8-accurate table built on the device with sincospi, staged in shared memory.  Sizes: 2^k (other
// 2^a 3^b 5^c 7^d sizes: fft_mixed.cu).
#include "fft_common.cuh"
#include <cuda.h>      // CUtensorMap types only: the encoder comes from cudaGetDriverEntryPoint (no -lcuda)
#include <map>
#include <mutex>
#include <tuple>
#include <stdlib.h>
#include <string.h>

// Stage plan: radix-8 stages, then one radix-4 or radix-2 stage for the remainder of log2(N).
// position (in the in-place DIF output) of frequency k = mixed-radix digit reversal
__device__ __forceinline__ int pos_of_freq(int k, int N, int log2n) {
    int rem = k, base = N, pos = 0;
    const int n8 = log2n / 3, r = log2n - 3 * n8;
    for (int s = 0; s < n8; s++) {
        int d = rem & 7;
        rem >>= 3;
        base >>= 3;
        pos += d * base;
    }
    if (r == 2) pos += (rem & 3);        // base == 4 -> base/4 == 1
    else if (r == 1) pos += (rem & 1);
    return pos;
}

// Shared-memory address (in elements) of line element e, column b.  Rows are padded to B+1 elements; with SKEW an
// extra element is inserted every N/8 rows, so that the digit-reversed rows 0, N/8, 2N/8, ... which consecutive
// output frequencies live in fall into different banks (the z passes read the tile with lanes along frequency).
template <int B, bool SKEW>
__device__ __forceinline__ int saddr(int e, int sk) { return e * (B + 1) + (SKEW ? (e >> sk) : 0); }

// In-place forward DIF FFT of B side-by-side lines of length N held at sm[saddr(n) + b].
// tw[k] = exp(-2 pi i k / N), k < N (shared or global memory).  All threads of the CTA must call.
// Each radix-8 butterfly lives in registers: 8 LDS + 8 STS per 8 points per stage (3 stages at N = 512).
template <typename C, int B, bool SKEW = false>
__device__ __forceinline__ void fft_tile(C *sm, const C *__restrict__ tw, int N, int log2n) {
    const int T = blockDim.x;
    const int sk = log2n >= 3 ? log2n - 3 : 31;
    const int n8 = log2n / 3, rrem = log2n - 3 * n8;
    int Ns = N;
    int lq = log2n;
    for (int s = 0; s < n8; s++) {
        const int Q = Ns >> 3;
        lq -= 3;                       // log2(Q)
        const int tws = N / Ns;
        const int work = (N >> 3) * B;
        for (int w = threadIdx.x; w < work; w += T) {
            int b = w % B;
            int t = w / B;
            int blk = t >> lq, q = t & (Q - 1);
            const int e0 = blk * Ns + q;
            C *p0 = sm + saddr<B, SKEW>(e0, sk) + b, *p1 = sm + saddr<B, SKEW>(e0 + Q, sk) + b;
            C *p2 = sm + saddr<B, SKEW>(e0 + 2 * Q, sk) + b, *p3 = sm + saddr<B, SKEW>(e0 + 3 * Q, sk) + b;
            C *p4 = sm + saddr<B, SKEW>(e0 + 4 * Q, sk) + b, *p5 = sm + saddr<B, SKEW>(e0 + 5 * Q, sk) + b;
            C *p6 = sm + saddr<B, SKEW>(e0 + 6 * Q, sk) + b, *p7 = sm + saddr<B, SKEW>(e0 + 7 * Q, sk) + b;
            C a0 = *p0, a1 = *p1, a2 = *p2, a3 = *p3, a4 = *p4, a5 = *p5, a6 = *p6, a7 = *p7;
            // level 1: b_m = a_m + a_{m+4}; b_{m+4} = (a_m - a_{m+4}) W8^m
            C b0 = cadd(a0, a4), b1 = cadd(a1, a5), b2 = cadd(a2, a6), b3 = cadd(a3, a7);
            C b4 = csub(a0, a4), d5 = csub(a1, a5), d6 = csub(a2, a6), d7 = csub(a3, a7);
            const auto h = Sqrt1_2<C>::v();
            C b5 = C{(d5.x + d5.y) * h, (d5.y - d5.x) * h};     // * (1 - i)/sqrt2
            C b6 = cmuli_neg(d6);                                // * (-i)
            C b7 = C{(d7.y - d7.x) * h, -(d7.x + d7.y) * h};    // * (-1 - i)/sqrt2
            dft4(b0, b1, b2, b3);      // -> y0, y2, y4, y6
            dft4(b4, b5, b6, b7);      // -> y1, y3, y5, y7
            if (Q > 1) {
                int ti = q * tws;
                b4 = cmul(b4, tw[ti]);
                b1 = cmul(b1, tw[2 * ti]);
                b5 = cmul(b5, tw[3 * ti]);
                b2 = cmul(b2, tw[4 * ti]);
                b6 = cmul(b6, tw[5 * ti]);
                b3 = cmul(b3, tw[6 * ti]);
                b7 = cmul(b7, tw[7 * ti]);
            }
            *p0 = b0; *p1 = b4; *p2 = b1; *p3 = b5; *p4 = b2; *p5 = b6; *p6 = b3; *p7 = b7;
        }
        __syncthreads();
        Ns = Q;
    }
    if (rrem == 2) {   // Ns == 4, Q == 1: no twiddles
        const int work = (N >> 2) * B;
        for (int w = threadIdx.x; w < work; w += T) {
            int b = w % B;
            int t = w / B;
            C *p0 = sm + saddr<B, SKEW>(4 * t, sk) + b, *p1 = sm + saddr<B, SKEW>(4 * t + 1, sk) + b;
            C *p2 = sm + saddr<B, SKEW>(4 * t + 2, sk) + b, *p3 = sm + saddr<B, SKEW>(4 * t + 3, sk) + b;
            C a0 = *p0, a1 = *p1, a2 = *p2, a3 = *p3;
            dft4(a0, a1, a2, a3);
            *p0 = a0; *p1 = a1; *p2 = a2; *p3 = a3;
        }
        __syncthreads();
    } else if (rrem == 1) {  // Ns == 2
        const int work = (N >> 1) * B;
        for (int w = threadIdx.x; w < work; w += T) {
            int b = w % B;
            int t = w / B;
            C *p0 = sm + saddr<B, SKEW>(2 * t, sk) + b, *p1 = sm + saddr<B, SKEW>(2 * t + 1, sk) + b;
            C a0 = *p0, a1 = *p1;
            *p0 = cadd(a0, a1);
            *p1 = csub(a0, a1);
        }
        __syncthreads();
    }
}

// copy the twiddle table into shared memory (after the tile); returns the shared pointer
template <typename C>
__device__ __forceinline__ const C *stage_twiddles(C *dst, const C *__restrict__ tw, int N) {
    for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = tw[i];
    __syncthreads();
    return dst;
}

// ---------------------------------------------------------------------------------------------
// strided line pass (y and x passes), in place.  element(outer, n, inner) =
//   data[outer*outer_stride + n*line_stride + inner],  inner < n_inner contiguous.
// ---------------------------------------------------------------------------------------------
// 16- / 8-byte asynchronous global -> shared copies (LDGSTS): the next tile streams in while this one is transformed
__device__ __forceinline__ void cp_async_elem(double2 *sdst, const double2 *gsrc) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_elem(float2 *sdst, const float2 *gsrc) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N_) : "memory"); }

// strided tile -> shared [N][B+1]; columns beyond the valid width are zero-filled with plain stores
template <typename C, int B>
__device__ __forceinline__ void prefetch_tile(C *sm, const C *base, int N, int64_t line_stride, int bvalid) {
    constexpr int pitch = B + 1;
    for (int w = threadIdx.x; w < N * B; w += blockDim.x) {
        int b = w % B, n = w / B;
        if (b < bvalid) cp_async_elem(&sm[n * pitch + b], base + (int64_t)n * line_stride + b);
        else sm[n * pitch + b] = C{0, 0};
    }
}

template <typename T, int B>
__global__ void __launch_bounds__(512)
k_fft_lines(const typename C2<T>::type *src, typename C2<T>::type *dst, const typename C2<T>::type *__restrict__ tw,
            int N, int log2n, int64_t line_stride, int64_t n_inner, int64_t tiles_inner, int64_t n_tiles, int64_t outer_stride,
            int inverse, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // shared: buf[2][N][B+1] | twiddles[N]  -- two tile buffers: tile i+1 is prefetched with cp.async while tile i is
    // transformed and written back
    C *buf0 = reinterpret_cast<C *>(smem_raw);
    constexpr int pitch = B + 1;
    C *buf1 = buf0 + (size_t)N * pitch;
    const int T_ = blockDim.x;
    tw = stage_twiddles<C>(buf1 + (size_t)N * pitch, tw, N);
    int64_t tile = blockIdx.x;
    if (tile < n_tiles) {
        int64_t outer = tile / tiles_inner;
        int64_t inner0 = (tile - outer * tiles_inner) * B;
        int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        prefetch_tile<C, B>(buf0, src + outer * outer_stride + inner0, N, line_stride, bvalid);
    }
    cp_async_commit();
    int cur = 0;
    for (; tile < n_tiles; tile += gridDim.x, cur ^= 1) {
        C *sm = cur ? buf1 : buf0;
        int64_t outer = tile / tiles_inner;
        int64_t inner0 = (tile - outer * tiles_inner) * B;
        C *obase = dst + outer * outer_stride + inner0;      // dst == src: in place (a CTA owns its tile)
        int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        int64_t nxt = tile + gridDim.x;
        if (nxt < n_tiles) {
            int64_t o2 = nxt / tiles_inner;
            int64_t i2 = (nxt - o2 * tiles_inner) * B;
            int bv2 = (int)((n_inner - i2) < B ? (n_inner - i2) : B);
            prefetch_tile<C, B>(cur ? buf0 : buf1, src + o2 * outer_stride + i2, N, line_stride, bv2);
        }
        cp_async_commit();
        cp_async_wait<1>();          // this tile's copies have landed (the prefetch may still be in flight)
        __syncthreads();
        if (inverse) {
            for (int w = threadIdx.x; w < N * B; w += T_) { int b = w % B, n = w / B; sm[n * pitch + b].y = -sm[n * pitch + b].y; }
            __syncthreads();
        }
        fft_tile<C, B>(sm, tw, N, log2n);
        for (int w = threadIdx.x; w < N * B; w += T_) {
            int b = w % B, k = w / B;
            if (b < bvalid) {
                C v = sm[pos_of_freq(k, N, log2n) * pitch + b];
                if (inverse) v.y = -v.y;
                v.x *= scale;
                v.y *= scale;
                obase[(int64_t)k * line_stride + b] = v;
            }
        }
        __syncthreads();             // everyone is done with `sm` before the next prefetch overwrites it
    }
    cp_async_wait<0>();
}
// ---------------------------------------------------------------------------------------------
// Fused line pass + slab transpose over peer memory (P > 1).  Lines of length N run along the SECOND stored axis
// of the local slab src[n_outer][N][n_inner] (the y pass of r2c on [x_n][Ny][Nzc], or the inverse x pass of c2r on
// [y_n][Nx][Nzc]).  Output frequency k belongs to rank p = k / (N/P); instead of writing the slab back, packing,
// all-to-all and unpacking, the store phase writes each 64..128-byte kz run straight into rank p's transposed
// field through its NVLink-mapped pointer:
//     peer[p][ ((k % (N/P)) * (n_outer*P) + outer_start + outer) * n_inner + kz ]
// (peer[rank] is the local buffer).  The caller brackets the launch with cross-rank barriers.
// ---------------------------------------------------------------------------------------------
#define NBK_MAX_PEERS 16
template <typename C> struct PeerPtrs { C *p[NBK_MAX_PEERS]; };

template <typename T, int B>
__global__ void __launch_bounds__(256)
k_fft_lines_scatter(const typename C2<T>::type *__restrict__ src, PeerPtrs<typename C2<T>::type> peers,
                    const typename C2<T>::type *__restrict__ tw, int N, int log2n, int64_t n_inner, int64_t tiles_inner,
                    int64_t n_tiles, int n_per, int64_t d_total, int64_t outer_start, int inverse, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    constexpr int pitch = B + 1;
    const int T_ = blockDim.x;
    tw = stage_twiddles<C>(sm + N * pitch, tw, N);
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int64_t outer = tile / tiles_inner;
        int64_t inner0 = (tile - outer * tiles_inner) * B;
        const C *base = src + outer * (int64_t)N * n_inner + inner0;
        int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        for (int w = threadIdx.x; w < N * B; w += T_) {
            int b = w % B, n = w / B;
            C v = C{0, 0};
            if (b < bvalid) v = base[(int64_t)n * n_inner + b];
            if (inverse) v.y = -v.y;
            sm[n * pitch + b] = v;
        }
        __syncthreads();
        fft_tile<C, B>(sm, tw, N, log2n);
        for (int w = threadIdx.x; w < N * B; w += T_) {
            int b = w % B, k = w / B;
            if (b < bvalid) {
                C v = sm[pos_of_freq(k, N, log2n) * pitch + b];
                if (inverse) v.y = -v.y;
                v.x *= scale;
                v.y *= scale;
                int p = k / n_per, kl = k - p * n_per;
                peers.p[p][((int64_t)kl * d_total + outer_start + outer) * n_inner + inner0 + b] = v;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Register-I/O line pass (N >= 64).  The first radix-8 stage loads its 8 inputs per butterfly straight from global
// memory (rows q + k*N/8, B adjacent columns per row = one 128-byte run per quarter warp), and the last stage
// writes its outputs straight to their digit-reversed frequency rows; shared memory only carries the exchanges
// between stages (4 instead of 8 shared accesses per element at N = 512, and no copy loops).  One tile buffer per
// CTA, so 2-3 CTAs share an SM and one CTA's global phase overlaps another's butterflies.
// PEER: the store goes to the NVLink-mapped transposed field of rank k / n_per (see k_fft_lines_scatter).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int rev8(int t, int ndig) {   // reverse the ndig base-8 digits of t
    int r = 0;
    for (int i = 0; i < ndig; i++) { r = (r << 3) | (t & 7); t >>= 3; }
    return r;
}

template <typename T, int B, bool PEER, int NT>
__global__ void __launch_bounds__(NT, 512 / NT)
k_fft_lines_rg(const typename C2<T>::type *src, typename C2<T>::type *dst, PeerPtrs<typename C2<T>::type> peers,
               const typename C2<T>::type *__restrict__ tw, int N, int log2n, int64_t line_stride, int64_t n_inner,
               int64_t tiles_inner, int64_t n_tiles, int64_t outer_stride, int n_per, int64_t d_total,
               int64_t outer_start, int inverse, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    constexpr int pitch = B + 1;
    const int T_ = blockDim.x;
    tw = stage_twiddles<C>(sm + (size_t)N * pitch, tw, N);
    const int n8 = log2n / 3, rrem = log2n - 3 * n8;
    const int Q1 = N >> 3;
    const T sgn = inverse ? (T)-1 : (T)1;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int64_t outer = tile / tiles_inner;
        int64_t inner0 = (tile - outer * tiles_inner) * B;
        const C *ibase = src + outer * outer_stride + inner0;
        int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        // ---- first stage: global -> registers -> shared
        for (int w = threadIdx.x; w < Q1 * B; w += T_) {
            int b = w % B, q = w / B;
            C a[8];
            if (b < bvalid) {
                const C *g = ibase + (int64_t)q * line_stride + b;
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = g[(int64_t)j * Q1 * line_stride];
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = C{0, 0};
            }
#pragma unroll
            for (int j = 0; j < 8; j++) a[j].y *= sgn;
            radix8(a);
            C *o = sm + q * pitch + b;
            o[0] = a[0];
#pragma unroll
            for (int m = 1; m < 8; m++) o[m * Q1 * pitch] = cmul(a[m], tw[m * q]);
        }
        __syncthreads();
        // ---- middle stages, in place in shared memory
        {
            const int last8 = rrem ? n8 : n8 - 1;    // radix-8 stages [1, last8) are exchanged through shared memory
            int Ns = Q1, lq = log2n - 3;
            for (int s = 1; s < last8; s++) {
                const int Q = Ns >> 3;
                lq -= 3;
                const int tws = N / Ns;
                for (int w = threadIdx.x; w < Q1 * B; w += T_) {
                    int b = w % B, t = w / B;
                    int blk = t >> lq, q = t & (Q - 1);
                    C *p = sm + (blk * Ns + q) * pitch + b;
                    C a[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) a[j] = p[j * Q * pitch];
                    radix8(a);
                    int ti = q * tws;
                    p[0] = a[0];
#pragma unroll
                    for (int m = 1; m < 8; m++) p[m * Q * pitch] = cmul(a[m], tw[m * ti]);
                }
                __syncthreads();
                Ns = Q;
            }
        }
        // ---- last stage: shared -> registers -> global (frequency rows)
        const int R = rrem == 0 ? 8 : (rrem == 2 ? 4 : 2);
        const int NR = N / R;                 // butterflies per line, and the frequency step between its outputs
        const int ndig = rrem == 0 ? n8 - 1 : n8;
        for (int w = threadIdx.x; w < NR * B; w += T_) {
            int b = w % B, t = w / B;
            const C *p = sm + (t * R) * pitch + b;
            C a[8];
            if (R == 8) {
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = p[j * pitch];
                radix8(a);
            } else if (R == 4) {
                a[0] = p[0]; a[1] = p[pitch]; a[2] = p[2 * pitch]; a[3] = p[3 * pitch];
                dft4(a[0], a[1], a[2], a[3]);
            } else {
                C x0 = p[0], x1 = p[pitch];
                a[0] = cadd(x0, x1);
                a[1] = csub(x0, x1);
            }
            if (b < bvalid) {
                int k0 = rev8(t, ndig);
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    if (m < R) {
                        int k = k0 + m * NR;
                        C v = C{a[m].x * scale, a[m].y * sgn * scale};
                        if (PEER) {
                            int pr = k / n_per, kl = k - pr * n_per;
                            peers.p[pr][((int64_t)kl * d_total + outer_start + outer) * n_inner + inner0 + b] = v;
                        } else {
                            dst[outer * outer_stride + inner0 + (int64_t)k * line_stride + b] = v;
                        }
                    }
                }
            }
        }
        __syncthreads();      // the next tile's first stage overwrites the buffer
    }
}

// ---------------------------------------------------------------------------------------------
// Register-I/O line pass with the NEXT tile's first-stage loads in flight during the last stage of the current one
// (ITER first-stage butterflies per thread, Q1 * B == ITER * NT).  With one 512-thread CTA per SM (lines of 1024
// complex doubles) nothing else hides the global-load latency: the loads of tile i+1 are issued before the last stage
// of tile i reads shared memory and streams its outputs out, so the memory system stays busy through the butterflies.
// ---------------------------------------------------------------------------------------------
template <typename T, int B, bool PEER, int NT, int ITER>
__global__ void __launch_bounds__(NT, 512 / NT)
k_fft_lines_rgp(const typename C2<T>::type *src, typename C2<T>::type *dst, PeerPtrs<typename C2<T>::type> peers,
                const typename C2<T>::type *__restrict__ tw, int N, int log2n, int64_t line_stride, int64_t n_inner,
                int64_t tiles_inner, int64_t n_tiles, int64_t outer_stride, int n_per, int64_t d_total,
                int64_t outer_start, int inverse, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    constexpr int pitch = B + 1;
    tw = stage_twiddles<C>(sm + (size_t)N * pitch, tw, N);
    const int n8 = log2n / 3, rrem = log2n - 3 * n8;
    const int Q1 = N >> 3;
    const T sgn = inverse ? (T)-1 : (T)1;
    C pre[ITER][8];
    auto issue_loads = [&](int64_t tile) {
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        const C *ibase = src + outer * outer_stride + inner0;
        const int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
#pragma unroll
        for (int it = 0; it < ITER; it++) {
            const int w = (int)threadIdx.x + it * NT;
            const int b = w % B, q = w / B;
            if (b < bvalid) {
                const C *g = ibase + (int64_t)q * line_stride + b;
#pragma unroll
                for (int j = 0; j < 8; j++) pre[it][j] = g[(int64_t)j * Q1 * line_stride];
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) pre[it][j] = C{0, 0};
            }
        }
    };
    int64_t tile = blockIdx.x;
    if (tile < n_tiles) issue_loads(tile);
    for (; tile < n_tiles; tile += gridDim.x) {
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        const int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        // ---- first stage: registers -> shared
#pragma unroll
        for (int it = 0; it < ITER; it++) {
            const int w = (int)threadIdx.x + it * NT;
            const int b = w % B, q = w / B;
            C a[8];
#pragma unroll
            for (int j = 0; j < 8; j++) { a[j] = pre[it][j]; a[j].y *= sgn; }
            radix8(a);
            C *o = sm + q * pitch + b;
            o[0] = a[0];
#pragma unroll
            for (int m = 1; m < 8; m++) o[m * Q1 * pitch] = cmul(a[m], tw[m * q]);
        }
        __syncthreads();
        // ---- middle stages, in place in shared memory
        {
            const int last8 = rrem ? n8 : n8 - 1;
            int Ns = Q1, lq = log2n - 3;
            for (int s = 1; s < last8; s++) {
                const int Q = Ns >> 3;
                lq -= 3;
                const int tws = N / Ns;
                for (int w = threadIdx.x; w < Q1 * B; w += NT) {
                    int b = w % B, t = w / B;
                    int blk = t >> lq, q = t & (Q - 1);
                    C *p = sm + (blk * Ns + q) * pitch + b;
                    C a[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) a[j] = p[j * Q * pitch];
                    radix8(a);
                    int ti = q * tws;
                    p[0] = a[0];
#pragma unroll
                    for (int m = 1; m < 8; m++) p[m * Q * pitch] = cmul(a[m], tw[m * ti]);
                }
                __syncthreads();
                Ns = Q;
            }
        }
        // ---- the next tile's inputs start travelling now
        if (tile + gridDim.x < n_tiles) issue_loads(tile + gridDim.x);
        // ---- last stage: shared -> registers -> global (frequency rows)
        const int R = rrem == 0 ? 8 : (rrem == 2 ? 4 : 2);
        const int NR = N / R;
        const int ndig = rrem == 0 ? n8 - 1 : n8;
        for (int w = threadIdx.x; w < NR * B; w += NT) {
            int b = w % B, t = w / B;
            const C *p = sm + (t * R) * pitch + b;
            C a[8];
            if (R == 8) {
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = p[j * pitch];
                radix8(a);
            } else if (R == 4) {
                a[0] = p[0]; a[1] = p[pitch]; a[2] = p[2 * pitch]; a[3] = p[3 * pitch];
                dft4(a[0], a[1], a[2], a[3]);
            } else {
                C x0 = p[0], x1 = p[pitch];
                a[0] = cadd(x0, x1);
                a[1] = csub(x0, x1);
            }
            if (b < bvalid) {
                int k0 = rev8(t, ndig);
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    if (m < R) {
                        int k = k0 + m * NR;
                        C v = C{a[m].x * scale, a[m].y * sgn * scale};
                        if (PEER) {
                            int pr = k / n_per, kl = k - pr * n_per;
                            peers.p[pr][((int64_t)kl * d_total + outer_start + outer) * n_inner + inner0 + b] = v;
                        } else {
                            dst[outer * outer_stride + inner0 + (int64_t)k * line_stride + b] = v;
                        }
                    }
                }
            }
        }
        __syncthreads();      // the next tile's first stage overwrites the buffer
    }
}

// ---------------------------------------------------------------------------------------------
// TMA-pipelined line pass (N = 64 R, R in {4, 8, 16}: lines of 256 / 512 / 1024).  Decimation in TIME over the first
// factor: the line x[n], n = j + R i, splits into R "row groups" j (rows j, j + R, ...: 64 rows of B adjacent columns =
// one 8 KB box of a 4-D tensor map {inner, j, i, outer}), each an independent 64-point FFT, followed by ONE radix-R
// combine  X[k + 64 m] = sum_j W_R^{jm} (W_N^{jk} Y_j[k]).
//   * one elected thread streams the groups of this CTA's tiles through a ring of NS = R + P shared-memory slots with
//     `cp.async.bulk.tensor` (SASS UTMALDG) + one mbarrier per slot: P groups of the NEXT tile are already in flight
//     while this tile is combined, the rest follow as soon as its slots are free -- the copy engine, not the warps'
//     registers, hides the HBM latency, and the warps only run butterflies;
//   * warp w owns group w of the tile: it waits for its own mbarrier and runs the 64-point FFT (8 x 8, two radix-8
//     stages in place, __syncwarp between) while later groups are still landing;
//   * after one CTA barrier every thread combines R values (radix-R in registers, natural output order) and stores the
//     frequency rows k + 64 m straight to global memory (128-byte runs); a second CTA barrier frees the R slots.
// Slots are dense [64][B] with B * sizeof(complex) = 128 bytes, lanes run along the columns first, so every quarter
// warp touches one full 128-byte row: conflict-free without padding.  In place (dst == src) is safe: a tile's stores
// only touch its own rows / columns, which were read completely before its combine.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned fm_smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fm_mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(fm_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fm_mbar_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(fm_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fm_mbar_wait(uint64_t *bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "NBK_FM_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra NBK_FM_DONE;\n"
        "bra NBK_FM_WAIT;\n"
        "NBK_FM_DONE:\n"
        "}\n" :: "r"(fm_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fm_tma_load_4d(void *sdst, const CUtensorMap *tmap, int c0, int c1, int c2, int c3, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
                 :: "r"(fm_smem_u32(sdst)), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(fm_smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void fm_tma_prefetch_4d(const CUtensorMap *tmap, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];"
                 :: "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

template <typename C> struct W16c;      // cos(pi/8), sin(pi/8)
template <> struct W16c<float2> { static __device__ __forceinline__ float c() { return 0.92387953251128675613f; }
                                  static __device__ __forceinline__ float s() { return 0.38268343236508977173f; } };
template <> struct W16c<double2> { static __device__ __forceinline__ double c() { return 0.92387953251128675613; }
                                   static __device__ __forceinline__ double s() { return 0.38268343236508977173; } };

// 16-point forward DFT in registers, natural order in and out (4 x 4: n = 4 n1 + n2, k = k1 + 4 k2)
template <typename C>
__device__ __forceinline__ void dft16(C (&a)[16]) {
    const auto h = Sqrt1_2<C>::v();
    const auto c8 = W16c<C>::c(), s8 = W16c<C>::s();
    C y[4][4];                                   // y[n2][k1]
#pragma unroll
    for (int n2 = 0; n2 < 4; n2++) {
        C b0 = a[n2], b1 = a[4 + n2], b2 = a[8 + n2], b3 = a[12 + n2];
        dft4(b0, b1, b2, b3);
        y[n2][0] = b0; y[n2][1] = b1; y[n2][2] = b2; y[n2][3] = b3;
    }
    // twiddles W_16^{n2 k1}
    y[1][1] = cmul(y[1][1], C{c8, -s8});                                   // W^1
    y[1][2] = C{(y[1][2].x + y[1][2].y) * h, (y[1][2].y - y[1][2].x) * h};  // W^2 = (1 - i)/sqrt2
    y[1][3] = cmul(y[1][3], C{s8, -c8});                                   // W^3
    y[2][1] = C{(y[2][1].x + y[2][1].y) * h, (y[2][1].y - y[2][1].x) * h};  // W^2
    y[2][2] = cmuli_neg(y[2][2]);                                          // W^4 = -i
    y[2][3] = C{(y[2][3].y - y[2][3].x) * h, -(y[2][3].x + y[2][3].y) * h}; // W^6 = (-1 - i)/sqrt2
    y[3][1] = cmul(y[3][1], C{s8, -c8});                                   // W^3
    y[3][2] = C{(y[3][2].y - y[3][2].x) * h, -(y[3][2].x + y[3][2].y) * h}; // W^6
    y[3][3] = cmul(y[3][3], C{-c8, s8});                                   // W^9 = -W^1
#pragma unroll
    for (int k1 = 0; k1 < 4; k1++) {
        C b0 = y[0][k1], b1 = y[1][k1], b2 = y[2][k1], b3 = y[3][k1];
        dft4(b0, b1, b2, b3);
        a[k1] = b0; a[k1 + 4] = b1; a[k1 + 8] = b2; a[k1 + 12] = b3;
    }
}
template <int R, typename C> __device__ __forceinline__ void dftR(C (&a)[R]) {
    if constexpr (R == 16) dft16(a);
    else if constexpr (R == 8) radix8(a);
    else { static_assert(R == 4, "combine radix"); dft4(a[0], a[1], a[2], a[3]); }
}

template <typename T, int R, int B, int NT, bool PEER>
__global__ void __launch_bounds__(NT)
k_fft_lines_tma(const __grid_constant__ CUtensorMap tmap, typename C2<T>::type *dst, PeerPtrs<typename C2<T>::type> peers,
                const typename C2<T>::type *__restrict__ twg, int64_t line_stride, int64_t n_inner, int64_t tiles_inner,
                int64_t n_tiles, int64_t outer_stride, int n_per, int64_t d_total, int64_t outer_start, int inverse, T scale,
                int NS, int l2_ahead) {
    typedef typename C2<T>::type C;
    // B side-by-side lines: 128-byte rows (8 c16 / 16 c8), or 64-byte rows at N = 1024 so that TWO CTAs share an SM
    constexpr int S = 64, N = S * R, NW = NT / 32, SLOT = S * B;
    static_assert((8 * B) % 32 == 0 && R % NW == 0, "tile geometry");
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    C *ring = reinterpret_cast<C *>(smem_raw);                 // [NS][64][B]
    C *twN = ring + (size_t)NS * SLOT;                         // W_N^i, i < N
    C *tw64 = twN + N;                                         // W_64^i, i < 64
    uint64_t *bars = reinterpret_cast<uint64_t *>(tw64 + S);   // [NS]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        for (int i = 0; i < NS; i++) fm_mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < N; i += NT) twN[i] = twg[i];
    for (int i = tid; i < S; i += NT) tw64[i] = twg[i * R];
    __syncthreads();
    const int64_t first = blockIdx.x;
    const int my_tiles = first < n_tiles ? (int)((n_tiles - first + gridDim.x - 1) / gridDim.x) : 0;
    const int G = my_tiles * R;                                // row groups this CTA streams
    const T sgn = inverse ? (T)-1 : (T)1;
    int issued = 0;
    auto issue = [&](int g) {
        const int it = g / R, j = g - it * R;
        const int64_t tile = first + (int64_t)it * gridDim.x;
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        const int slot = g % NS;
        fm_mbar_expect_tx(&bars[slot], (unsigned)(SLOT * sizeof(C)));
        fm_tma_load_4d(ring + (size_t)slot * SLOT, &tmap, (int)(2 * inner0), j, 0, (int)outer, &bars[slot]);
    };
    // optional (l2_ahead, off by default: measured slower): L2 prefetch of the boxes one tile beyond what the ring can hold
    int fetched = 0;
    auto prefetch = [&](int g) {
        const int it = g / R, j = g - it * R;
        const int64_t tile = first + (int64_t)it * gridDim.x;
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        fm_tma_prefetch_4d(&tmap, (int)(2 * inner0), j, 0, (int)outer);
    };
    if (tid == 0) {
        const int upto = G < NS ? G : NS;
        for (; issued < upto; issued++) issue(issued);
        if (l2_ahead) {
            int pf = issued + R < G ? issued + R : G;
            for (fetched = issued; fetched < pf; fetched++) prefetch(fetched);
        }
    }
    for (int it = 0; it < my_tiles; it++) {
        const int64_t tile = first + (int64_t)it * gridDim.x;
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        const int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        // ---- 64-point FFT of my row group (warp-local: two radix-8 stages in place)
        for (int gw = warp; gw < R; gw += NW) {
            const int g = it * R + gw, slot = g % NS;
            fm_mbar_wait(&bars[slot], (unsigned)((g / NS) & 1));
            C *sl = ring + (size_t)slot * SLOT;
            constexpr int IT = (8 * B) / 32;
#pragma unroll
            for (int i = 0; i < IT; i++) {
                const int w = lane + 32 * i, b = w % B, q = w / B;
                C *p = sl + q * B + b;
                C a[8];
#pragma unroll
                for (int j = 0; j < 8; j++) { a[j] = p[j * 8 * B]; a[j].y *= sgn; }
                radix8(a);
                p[0] = a[0];
#pragma unroll
                for (int m = 1; m < 8; m++) p[m * 8 * B] = cmul(a[m], tw64[m * q]);
            }
            __syncwarp();
#pragma unroll
            for (int i = 0; i < IT; i++) {
                const int w = lane + 32 * i, b = w % B, t = w / B;
                C *p = sl + t * 8 * B + b;
                C a[8];
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = p[j * B];
                radix8(a);
#pragma unroll
                for (int m = 0; m < 8; m++) p[m * B] = a[m];       // position 8 t + m holds frequency t + 8 m
            }
        }
        __syncthreads();
        // ---- radix-R combine across the groups, registers -> global frequency rows k + 64 m
        {
            const int base = (it * R) % NS;
            for (int w = tid; w < S * B; w += NT) {
                const int b = w % B, k = w / B;
                const int pos = ((k & 7) << 3) | (k >> 3);
                C a[R];
#pragma unroll
                for (int j = 0; j < R; j++) {
                    int sj = base + j;
                    if (sj >= NS) sj -= NS;
                    C v = ring[(size_t)sj * SLOT + pos * B + b];
                    a[j] = j ? cmul(v, twN[j * k]) : v;
                }
                dftR<R, C>(a);
                if (b < bvalid) {
#pragma unroll
                    for (int m = 0; m < R; m++) {
                        const int K = k + S * m;
                        const C v = C{a[m].x * scale, a[m].y * sgn * scale};
                        if (PEER) {
                            const int pr = K / n_per, kl = K - pr * n_per;
                            peers.p[pr][((int64_t)kl * d_total + outer_start + outer) * n_inner + inner0 + b] = v;
                        } else {
                            dst[outer * outer_stride + inner0 + (int64_t)K * line_stride + b] = v;
                        }
                    }
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic accesses to the slots before the next TMA writes
        __syncthreads();
        if (tid == 0) {
            int upto = (it + 1) * R + NS;
            if (upto > G) upto = G;
            for (; issued < upto; issued++) issue(issued);
            if (l2_ahead) {
                int pf = issued + R < G ? issued + R : G;
                if (fetched < issued) fetched = issued;
                for (; fetched < pf; fetched++) prefetch(fetched);
            }
        }
    }
}

typedef CUresult (*nbk_encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                        const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static nbk_encode_tiled_fn get_tensor_map_encoder() {
    static std::mutex m;
    static bool tried = false;
    static nbk_encode_tiled_fn fn = nullptr;
    std::lock_guard<std::mutex> lock(m);
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (nbk_encode_tiled_fn)p;
        else
            (void)cudaGetLastError();
    }
    return fn;
}

// ---------------------------------------------------------------------------------------------
// z pass forward: real rows [rows][Nz] -> complex rows [rows][Nz/2+1]
// packed trick: z[n] = x[2n] + i x[2n+1], Z = FFT_M(z), M = Nz/2,
//   X[k] = 1/2 [ (Z[k] + conj Z[M-k]) - i W_N^k (Z[k] - conj Z[M-k]) ],  k = 0..M  (Z[M] := Z[0])
// ---------------------------------------------------------------------------------------------
template <typename T, int B>
__global__ void __launch_bounds__(256)
k_fft_z_r2c(const T *__restrict__ real, typename C2<T>::type *__restrict__ cplx,
            const typename C2<T>::type *__restrict__ twM, const typename C2<T>::type *__restrict__ twN, int Nz,
            int log2m, int64_t rows, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const int M = Nz >> 1;
    const int Nzc = M + 1;
    constexpr int pitch = B + 1;
    const int T_ = blockDim.x;
    const int sk = log2m >= 3 ? log2m - 3 : 31;
    const int64_t n_tiles = (rows + B - 1) / B;
    twM = stage_twiddles<C>(sm + M * pitch + 8, twM, M);
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int64_t row0 = tile * B;
        int bvalid = (int)((rows - row0) < B ? (rows - row0) : B);
        const C *src = reinterpret_cast<const C *>(real + row0 * Nz);  // rows of M packed pairs, 2*sizeof(T) aligned
        for (int w = threadIdx.x; w < M * B; w += T_) {
            int n = w & (M - 1), b = w >> log2m;  // lanes run along the contiguous row
            C v = C{0, 0};
            if (b < bvalid) v = src[(int64_t)b * M + n];
            sm[saddr<B, true>(n, sk) + b] = v;
        }
        __syncthreads();
        fft_tile<C, B, true>(sm, twM, M, log2m);
        C *dst = cplx + row0 * Nzc;
        for (int w = threadIdx.x; w < Nzc * B; w += T_) {
            int k = w % Nzc, b = w / Nzc;
            if (b < bvalid) {
                C zk = sm[saddr<B, true>(pos_of_freq(k & (M - 1), M, log2m), sk) + b];
                C zm = cconj(sm[saddr<B, true>(pos_of_freq((M - k) & (M - 1), M, log2m), sk) + b]);
                dst[(int64_t)b * Nzc + k] = hermitian_split(zk, zm, twN[k], (T)0.5 * scale);
            }
        }
        __syncthreads();
    }
}

// Last DIF stage of B side-by-side length-M lines in shared memory, leaving the spectrum in NATURAL order: every thread
// first pulls all of its butterflies into registers (V values: M * B <= 256 V; V = 16 for c8, 8 for c16 keeps them in 32 registers), then the CTA
// synchronises, then the outputs are stored at their frequency rows.
template <typename C, int B, int R, int V>
__device__ __forceinline__ void last_stage_natural(C *sm, int M, int ndig) {
    constexpr int pitch = B + 1;
    constexpr int NB = V / R;
    const int NR = M / R;
    C a[NB][R];
#pragma unroll
    for (int it = 0; it < NB; it++) {
        int w = threadIdx.x + it * 256;
        if (w < NR * B) {
            int b = w % B, t = w / B;
            const C *p = sm + (t * R) * pitch + b;
#pragma unroll
            for (int j = 0; j < R; j++) a[it][j] = p[j * pitch];
            if constexpr (R == 8) {
                radix8(a[it]);
            } else if constexpr (R == 4) {
                dft4(a[it][0], a[it][1], a[it][2], a[it][3]);
            } else {
                C x0 = a[it][0], x1 = a[it][1];
                a[it][0] = cadd(x0, x1);
                a[it][1] = csub(x0, x1);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < NB; it++) {
        int w = threadIdx.x + it * 256;
        if (w < NR * B) {
            int b = w % B, t = w / B;
            int k0 = rev8(t, ndig);
#pragma unroll
            for (int m = 0; m < R; m++) sm[(k0 + m * NR) * pitch + b] = a[it][m];
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// z pass forward, register-I/O variant (Nz >= 128).  Same packed-pair algorithm as k_fft_z_r2c; the first radix-8
// stage reads the real row straight from global memory (lanes along the row: 512-byte runs), the last stage leaves
// Z in NATURAL frequency order in shared memory (registers carry the permutation across one barrier), so the
// Hermitian split reads Z[k] and Z[M-k] with unit-stride lanes and no digit-reversal arithmetic.  Shared: tile
// [M][B+1] | W_N table [N] (W_M^j = W_N^2j serves the butterflies, W_N^k the split) | first-stage twiddles [7][M/8].
// ---------------------------------------------------------------------------------------------
template <typename T, int B>
__global__ void __launch_bounds__(256, 2)
k_fft_z_r2c_rg(const T *__restrict__ real, typename C2<T>::type *__restrict__ cplx,
               const typename C2<T>::type *__restrict__ twN_g, int Nz, int log2m, int64_t rows, T scale) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const int M = Nz >> 1;
    const int Nzc = M + 1;
    constexpr int pitch = B + 1;
    const int T_ = blockDim.x;
    // first-stage twiddles transposed to [m][q] (lanes run along q there: unit stride instead of stride 2m)
    C *tw1 = sm + (size_t)M * pitch + Nz;
    for (int i = threadIdx.x; i < 7 * (M >> 3); i += blockDim.x) {
        int m = i / (M >> 3) + 1, q = i - (m - 1) * (M >> 3);
        tw1[i] = twN_g[2 * m * q];
    }
    const C *tw = stage_twiddles<C>(sm + (size_t)M * pitch, twN_g, Nz);    // tw[2j] = W_M^j
    const int n8 = log2m / 3, rrem = log2m - 3 * n8;
    const int Q1 = M >> 3, lq1 = log2m - 3;
    const int64_t n_tiles = (rows + B - 1) / B;
    const T h = (T)0.5 * scale;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * B;
        const int bvalid = (int)((rows - row0) < B ? (rows - row0) : B);
        const C *src = reinterpret_cast<const C *>(real + row0 * Nz);    // rows of M packed pairs
        // ---- first stage: global -> registers -> shared; lanes along the row
        for (int w = threadIdx.x; w < Q1 * B; w += T_) {
            int q = w & (Q1 - 1), b = w >> lq1;
            C a[8];
            if (b < bvalid) {
                const C *g = src + (int64_t)b * M + q;
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = g[j * Q1];
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = C{0, 0};
            }
            radix8(a);
            C *o = sm + q * pitch + b;
            o[0] = a[0];
#pragma unroll
            for (int m = 1; m < 8; m++) o[m * Q1 * pitch] = cmul(a[m], tw1[(m - 1) * Q1 + q]);
        }
        __syncthreads();
        // ---- middle stages, in place
        {
            const int last8 = rrem ? n8 : n8 - 1;
            int Ns = Q1, lq = lq1;
            for (int s = 1; s < last8; s++) {
                const int Q = Ns >> 3;
                lq -= 3;
                const int tws = 2 * (M / Ns);
                for (int w = threadIdx.x; w < Q1 * B; w += T_) {
                    int b = w % B, t = w / B;
                    int blk = t >> lq, q = t & (Q - 1);
                    C *p = sm + (blk * Ns + q) * pitch + b;
                    C a[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) a[j] = p[j * Q * pitch];
                    radix8(a);
                    int ti = q * tws;
                    p[0] = a[0];
#pragma unroll
                    for (int m = 1; m < 8; m++) p[m * Q * pitch] = cmul(a[m], tw[m * ti]);
                }
                __syncthreads();
                Ns = Q;
            }
        }
        // ---- last stage: all M*B/256 <= V values of a thread go to registers, barrier, natural-order write back
        constexpr int V = sizeof(T) == 4 ? 16 : 8;
        if (rrem == 0) last_stage_natural<C, B, 8, V>(sm, M, n8 - 1);
        else if (rrem == 2) last_stage_natural<C, B, 4, V>(sm, M, n8);
        else last_stage_natural<C, B, 2, V>(sm, M, n8);
        // ---- Hermitian split, one warp per row, lanes along k
        C *dst = cplx + row0 * Nzc;
        for (int b = threadIdx.x >> 5; b < bvalid; b += (T_ >> 5)) {
            C *drow = dst + (int64_t)b * Nzc;
            for (int k = threadIdx.x & 31; k < Nzc; k += 32) {
                C zk = sm[(k & (M - 1)) * pitch + b];
                C zm = cconj(sm[((M - k) & (M - 1)) * pitch + b]);
                C e = cadd(zk, zm), o = csub(zk, zm);
                C wo = cmul(tw[k], o);
                drow[k] = C{(e.x + wo.y) * h, (e.y - wo.x) * h};
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// z pass forward, warp-per-row with TMA bulk row copies (Nz = 2M, M in {128, 256, 512}).  Every warp owns a private ring of
// row buffers: one lane streams the next rows of the warp in with `cp.async.bulk` (one 1-D copy of the whole row, SASS
// UBLKCP) + an mbarrier per buffer while the warp transforms the row that has landed -- packed-pair M-point FFT (radix 8,
// 8, M/64, in place, __syncwarp between the stages), Hermitian split, coalesced stores of the Nz/2+1 modes.  No CTA
// barrier after the twiddle staging, so the warps of an SM drift apart and the loads never stop.
// Shared-memory positions are XOR-swizzled, pos(e) = e ^ ((e >> 3) & 7) (a permutation inside each aligned group of 8
// elements = one 128-byte line of c16), which makes the stride-8 accesses of the later stages and the natural-order
// write of the last stage bank-conflict free; the copy engine lands the row unswizzled and the first stage re-places it.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void fm_bulk_g2s(void *sdst, const void *gsrc, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(fm_smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(fm_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ int fm_sw(int e) { return e ^ ((e >> 3) & 7); }

template <typename T, int LM, int NW>
__global__ void __launch_bounds__(32 * NW)
k_fft_z_r2c_tma(const T *__restrict__ real, typename C2<T>::type *__restrict__ cplx,
                const typename C2<T>::type *__restrict__ twN_g, int64_t rows, T scale, int nbuf) {
    typedef typename C2<T>::type C;
    constexpr int M = 1 << LM, Nz = 2 * M, Nzc = M + 1;
    constexpr int R3 = M / 64;                    // last radix: 8 / 4 / 2
    constexpr int Q1 = M / 8;                     // butterflies of the radix-8 stages
    constexpr int I1 = (Q1 + 31) / 32;            // ... per lane
    extern __shared__ __align__(128) unsigned char smem_raw[];
    C *twN = reinterpret_cast<C *>(smem_raw);                         // W_N^i, i <= M  (Hermitian split)
    C *tw1 = twN + Nz;                                                // [7][Q1]  W_M^{q m}: lanes along q, unit stride
    C *tw2 = tw1 + 7 * Q1;                                            // [7][R3]  W_{8 R3}^{q m}
    C *bufs = tw2 + 7 * 8;                                            // [NW][nbuf][M]
    uint64_t *bars = reinterpret_cast<uint64_t *>(bufs + (size_t)NW * nbuf * M);   // [NW][nbuf]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < Nz; i += 32 * NW) twN[i] = twN_g[i];
    // (a strided twN[2 m q] / twN[16 m q] puts the lanes of a quarter warp on the same banks: 8-way conflicts that made
    // the twiddle reads cost more shared-memory wavefronts than the data)
    for (int i = threadIdx.x; i < 7 * Q1; i += 32 * NW) { const int m = i / Q1 + 1, q = i % Q1; tw1[i] = twN_g[2 * m * q]; }
    for (int i = threadIdx.x; i < 7 * R3; i += 32 * NW) { const int m = i / R3 + 1, q = i % R3; tw2[i] = twN_g[(16 * m * q) % Nz]; }
    if (lane == 0) {
        for (int i = 0; i < nbuf; i++) fm_mbar_init(&bars[warp * nbuf + i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t gw = (int64_t)blockIdx.x * NW + warp, GW = (int64_t)gridDim.x * NW;
    const int64_t my_rows = gw < rows ? (rows - gw + GW - 1) / GW : 0;
    C *wbuf = bufs + (size_t)warp * nbuf * M;
    uint64_t *wbar = bars + warp * nbuf;
    const unsigned row_bytes = (unsigned)(M * sizeof(C));
    auto issue = [&](int64_t i) {     // lane 0 only
        const int sidx = (int)(i % nbuf);
        fm_mbar_expect_tx(&wbar[sidx], row_bytes);
        fm_bulk_g2s(wbuf + (size_t)sidx * M, real + (gw + i * GW) * (int64_t)Nz, row_bytes, &wbar[sidx]);
    };
    if (lane == 0) for (int64_t i = 0; i < nbuf && i < my_rows; i++) issue(i);
    const T h = (T)0.5 * scale;
    for (int64_t i = 0; i < my_rows; i++) {
        const int sidx = (int)(i % nbuf);
        fm_mbar_wait(&wbar[sidx], (unsigned)((i / nbuf) & 1));
        C *z = wbuf + (size_t)sidx * M;
        // ---- stage 1 (radix 8 over elements q + Q1 j): reads the landed (unswizzled) row, writes swizzled
        {
            C a[I1][8];
#pragma unroll
            for (int it = 0; it < I1; it++) {
                const int q = lane + 32 * it;
                if (q < Q1) {
#pragma unroll
                    for (int j = 0; j < 8; j++) a[it][j] = z[q + Q1 * j];
                }
            }
            __syncwarp();
#pragma unroll
            for (int it = 0; it < I1; it++) {
                const int q = lane + 32 * it;
                if (q < Q1) {
                    radix8(a[it]);
                    z[fm_sw(q)] = a[it][0];
#pragma unroll
                    for (int m = 1; m < 8; m++) z[fm_sw(q + Q1 * m)] = cmul(a[it][m], tw1[(m - 1) * Q1 + q]);
                }
            }
        }
        __syncwarp();
        // ---- stage 2 (radix 8 inside the 8 blocks of Q1 elements: elements blk Q1 + q + R3 j), in place
#pragma unroll
        for (int it = 0; it < I1; it++) {
            const int t = lane + 32 * it;
            if (t < Q1) {
                const int blk = t / R3, q = t - blk * R3;
                const int e0 = blk * Q1 + q;
                C a[8];
#pragma unroll
                for (int j = 0; j < 8; j++) a[j] = z[fm_sw(e0 + R3 * j)];
                radix8(a);
                z[fm_sw(e0)] = a[0];
#pragma unroll
                for (int m = 1; m < 8; m++) z[fm_sw(e0 + R3 * m)] = cmul(a[m], tw2[(m - 1) * R3 + q]);      // W_{8 R3}^{q m}
            }
        }
        __syncwarp();
        // ---- stage 3 (radix R3 over elements R3 t + j, 64 butterflies); outputs go to NATURAL frequency positions:
        // position R3 t + m3 holds frequency (t / 8) + 8 (t % 8) + 64 m3
        {
            C a[2][R3];
#pragma unroll
            for (int it = 0; it < 2; it++) {
                const int t = lane + 32 * it;
#pragma unroll
                for (int j = 0; j < R3; j++) a[it][j] = z[fm_sw(R3 * t + j)];
            }
            __syncwarp();
#pragma unroll
            for (int it = 0; it < 2; it++) {
                const int t = lane + 32 * it;
                if constexpr (R3 == 8) radix8(a[it]);
                else if constexpr (R3 == 4) dft4(a[it][0], a[it][1], a[it][2], a[it][3]);
                else { C x0 = a[it][0], x1 = a[it][1]; a[it][0] = cadd(x0, x1); a[it][1] = csub(x0, x1); }
                const int k0 = (t >> 3) + 8 * (t & 7);
#pragma unroll
                for (int m = 0; m < R3; m++) z[fm_sw(k0 + 64 * m)] = a[it][m];
            }
        }
        __syncwarp();
        // ---- Hermitian split, lanes along k:  X[k] = 1/2 [ (Z[k] + conj Z[M-k]) - i W_N^k (Z[k] - conj Z[M-k]) ]
        C *drow = cplx + (gw + i * GW) * (int64_t)Nzc;
        for (int k = lane; k < Nzc; k += 32) {
            const C zk = z[fm_sw(k & (M - 1))];
            const C zm = cconj(z[fm_sw((M - k) & (M - 1))]);
            const C e = cadd(zk, zm), o = csub(zk, zm);
            const C wo = cmul(twN[k], o);
            drow[k] = C{(e.x + wo.y) * h, (e.y - wo.x) * h};
        }
        // ---- the buffer is free: fetch the row that will use it next
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0 && i + nbuf < my_rows) issue(i + nbuf);
    }
}

// z pass backward: complex rows [rows][Nz/2+1] -> real rows [rows][Nz], unnormalised
//   E = (X[k] + conj X[M-k])/2, O = conj(W_N^k) (X[k] - conj X[M-k])/2, Z[k] = E + i O, k < M
//   x[2n] + i x[2n+1] = 2 * sum_k Z[k] e^{+2 pi i k n / M} = 2 * conj(FFT_M(conj Z))[n]
template <typename T, int B>
__global__ void __launch_bounds__(256)
k_fft_z_c2r(const typename C2<T>::type *__restrict__ cplx, T *__restrict__ real,
            const typename C2<T>::type *__restrict__ twM, const typename C2<T>::type *__restrict__ twN, int Nz,
            int log2m, int64_t rows) {
    typedef typename C2<T>::type C;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const int M = Nz >> 1;
    const int Nzc = M + 1;
    constexpr int pitch = B + 1;
    const int T_ = blockDim.x;
    const int sk = log2m >= 3 ? log2m - 3 : 31;
    const int64_t n_tiles = (rows + B - 1) / B;
    twM = stage_twiddles<C>(sm + M * pitch + 8, twM, M);
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int64_t row0 = tile * B;
        int bvalid = (int)((rows - row0) < B ? (rows - row0) : B);
        const C *src = cplx + row0 * Nzc;
        for (int w = threadIdx.x; w < M * B; w += T_) {
            int k = w & (M - 1), b = w >> log2m;
            C v = C{0, 0};
            if (b < bvalid) {
                v = hermitian_merge(src[(int64_t)b * Nzc + k], cconj(src[(int64_t)b * Nzc + (M - k)]), twN[k]);
            }
            sm[saddr<B, true>(k, sk) + b] = v;
        }
        __syncthreads();
        fft_tile<C, B, true>(sm, twM, M, log2m);
        C *dst = reinterpret_cast<C *>(real + row0 * Nz);
        for (int w = threadIdx.x; w < M * B; w += T_) {
            int n = w & (M - 1), b = w >> log2m;
            if (b < bvalid) {
                C v = cconj(sm[saddr<B, true>(pos_of_freq(n, M, log2m), sk) + b]);
                dst[(int64_t)b * M + n] = v;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// twiddle tables, cached per (device, N, dtype)
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_twiddle(typename C2<T>::type *tw, int N) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < N) {
        double s, c;
        sincospi(-2.0 * (double)k / (double)N, &s, &c);
        tw[k].x = (T)c;
        tw[k].y = (T)s;
    }
}

static std::mutex g_tw_mutex;
static std::map<std::tuple<int, int, int>, void *> g_tw;

int get_twiddle(int N, int dtype, cudaStream_t s, void **out) {
    int dev = 0;
    NBK_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_tw_mutex);
    auto key = std::make_tuple(dev, N, dtype);
    auto it = g_tw.find(key);
    if (it != g_tw.end()) { *out = it->second; return NBK_OK; }
    void *p = nullptr;
    size_t bytes = (size_t)(N > 0 ? N : 1) * (dtype == NBK_F4 ? 8 : 16);
    NBK_CUDA(cudaMalloc(&p, bytes));
    int g = (N + 255) / 256;
    if (g < 1) g = 1;
    if (dtype == NBK_F4) k_twiddle<float><<<g, 256, 0, s>>>((float2 *)p, N);
    else k_twiddle<double><<<g, 256, 0, s>>>((double2 *)p, N);
    NBK_LAUNCHED();
    // table must be visible to later launches on other streams as well
    NBK_CUDA(cudaStreamSynchronize(s));
    g_tw[key] = p;
    *out = p;
    return NBK_OK;
}

static int ilog2(int64_t n) {
    int l = 0;
    while (((int64_t)1 << l) < n) l++;
    return l;
}
static bool is_pow2(int64_t n) { return n > 0 && (n & (n - 1)) == 0; }

// pick the number of side-by-side lines: >= 64 B contiguous runs, tile <= ~96 KB (2 CTAs / SM)
static int pick_B(int N, int csize, int64_t n_inner) {
    int B = 128 / csize;  // 128-byte runs: 16 (c8) or 8 (c16)
    while (B > 1 && (size_t)N * (B + 2) * csize > 98304) B >>= 1;
    while (B > 1 && B / 2 >= n_inner) B >>= 1;
    return B;
}

static bool use_reg_lines(int N) {
    static int mode = -1;
    if (mode < 0) {
        const char *e = getenv("NBK_FFT_LINES");
        mode = (e && strcmp(e, "smem") == 0) ? 0 : 1;      // "rg" / default: register-I/O family (the TMA pass is tried first)
    }
    return mode == 1 && N >= 64;
}

// TMA-pipelined line pass (k_fft_lines_tma) where it applies: N in {256, 512, 1024}, 16-byte aligned rows (always true
// for c16 fields; c8 fields with an odd row length -- the y pass over Nz/2+1 columns -- keep the register-I/O kernel).
// NBK_FFT_LINES=rg|smem selects the older kernels.  *done = false: not applicable, the caller falls back.
static int lines_mode() {
    static int mode = -1;
    if (mode < 0) {
        const char *e = getenv("NBK_FFT_LINES");
        mode = (e && strcmp(e, "smem") == 0) ? 0 : (e && strcmp(e, "rg") == 0) ? 1 : 2;
    }
    return mode;
}
template <typename T>
static int launch_lines_tma(const void *src, void *dst, void *const *peer_host, int P, int N, int64_t line_stride,
                            int64_t n_inner, int64_t n_outer, int64_t outer_stride, int64_t outer_start, int inverse,
                            double scale, cudaStream_t s, int64_t d_total_override, bool *done) {
    typedef typename C2<T>::type C;
    *done = false;
    if (lines_mode() != 2 || (N != 256 && N != 512 && N != 1024)) return NBK_OK;
    const size_t cs = sizeof(C);
    if (n_outer > 1 && outer_stride == 0) return NBK_OK;
    const int64_t ostride = n_outer > 1 ? outer_stride : (int64_t)N * line_stride;
    if ((reinterpret_cast<uintptr_t>(src) & 15) || ((size_t)line_stride * cs) % 16 || ((size_t)ostride * cs) % 16) return NBK_OK;
    if (2 * n_inner >= (1ll << 31) || n_outer >= (1ll << 31) || (size_t)ostride * cs >= ((size_t)1 << 40) ||
        (size_t)(N / 64) * line_stride * cs >= ((size_t)1 << 40)) return NBK_OK;
    nbk_encode_tiled_fn enc = get_tensor_map_encoder();
    if (!enc) return NBK_OK;
    const int R = N / 64;
    // tile width: 128-byte rows.  (64-byte rows -- half the ring, two CTAs per SM at N = 1024 -- are selectable with
    // NBK_FFT_TMA_B = columns; measured slower: the x pass of 1024^3 f8 takes 7.2 ms instead of 4.1.)
    static int knob_b = -1, knob_ns = -1, l2_ahead = -1;
    // NBK_FFT_TMA_L2=1: L2 tensor prefetch one tile ahead of the ring.  Off: measured SLOWER (1024^3 f8: y 4.22 -> 5.36 ms, x 4.07
    // -> 5.57 ms; 512^3: x 0.43 -> 0.61 ms) -- the prefetches compete with the demand loads and stores for DRAM.
    if (l2_ahead < 0) { const char *e = getenv("NBK_FFT_TMA_L2"); l2_ahead = (e && e[0] == '1') ? 1 : 0; }
    if (knob_b < 0) { const char *e = getenv("NBK_FFT_TMA_B"); knob_b = e ? atoi(e) : 0; }
    if (knob_ns < 0) { const char *e = getenv("NBK_FFT_TMA_NS"); knob_ns = e ? atoi(e) : 0; }
    const int Bfull = 128 / (int)cs;
    int B = Bfull;
    if (N != 256 && (knob_b == Bfull || knob_b == Bfull / 2)) B = knob_b;
    CUtensorMap tmap;
    const cuuint64_t gdim[4] = {(cuuint64_t)(2 * n_inner), (cuuint64_t)R, 64, (cuuint64_t)n_outer};
    const cuuint64_t gstr[3] = {(cuuint64_t)line_stride * cs, (cuuint64_t)R * line_stride * cs, (cuuint64_t)ostride * cs};
    const cuuint32_t box[4] = {(cuuint32_t)(2 * B), 1, 64, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult cr = enc(&tmap, sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4,
                      const_cast<void *>(src), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return NBK_OK;                     // shape the encoder refuses: older kernels
    int dtype = sizeof(T) == 4 ? NBK_F4 : NBK_F8;
    void *tw;
    int rc = get_twiddle(N, dtype, s, &tw);
    if (rc) return rc;
    // ring: R slots of the tile being transformed + P prefetch slots, sized for 2 CTAs / SM (3 at N = 256); the wide
    // tile at N = 1024 takes the whole SM
    const size_t slot = (size_t)64 * B * cs;
    const size_t fixed = (size_t)(N + 64) * cs + 26 * 8 + 64;
    int per_sm = (R == 16 && B == Bfull) ? 1 : (R == 4 ? 3 : 2);
    int NS = (int)(((size_t)(226 * 1024) / per_sm - 1024 - fixed) / slot);
    if (NS > 26) NS = 26;
    if (NS > 2 * R) NS = 2 * R;
    if (knob_ns >= R + 1 && knob_ns <= NS) NS = knob_ns;
    NBK_CHECK_ARG(NS >= R + 1, "fft_lines: the slot ring does not fit in shared memory (N = %d)", N);
    const size_t smem = (size_t)NS * slot + fixed;
    const int64_t tiles_inner = (n_inner + B - 1) / B;
    const int64_t n_tiles = tiles_inner * n_outer;
    const int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
    PeerPtrs<C> peers;
    for (int i = 0; i < NBK_MAX_PEERS; i++) peers.p[i] = (peer_host && i < P) ? (C *)peer_host[i] : nullptr;
    const int n_per = peer_host ? N / P : N;
    const int64_t d_total = d_total_override ? d_total_override : (peer_host ? n_outer * P : 0);
#define LAUNCH_TMA2(RR, BB, NTT, PEERF)                                                                                \
    do {                                                                                                               \
        NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_tma<T, RR, BB, NTT, PEERF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_fft_lines_tma<T, RR, BB, NTT, PEERF><<<(int)g, NTT, smem, s>>>(tmap, (C *)dst, peers, (const C *)tw, line_stride, n_inner, \
            tiles_inner, n_tiles, outer_stride, n_per, d_total, outer_start, inverse, (T)scale, NS, l2_ahead);        \
    } while (0)
#define LAUNCH_TMA(RR, BB, NTT) do { if (peer_host) LAUNCH_TMA2(RR, BB, NTT, true); else LAUNCH_TMA2(RR, BB, NTT, false); } while (0)
    constexpr int BF = 128 / (int)sizeof(C), BH = BF / 2;
    if (R == 16 && B == BF) LAUNCH_TMA(16, BF, 512);
    else if (R == 16) LAUNCH_TMA(16, BH, 256);
    else if (R == 8 && B == BF) LAUNCH_TMA(8, BF, 256);
    else if (R == 8) LAUNCH_TMA(8, BH, 256);
    else LAUNCH_TMA(4, BF, 128);
#undef LAUNCH_TMA
#undef LAUNCH_TMA2
    NBK_LAUNCHED();
    *done = true;
    return NBK_OK;
}

// register-I/O line pass; peer_host != nullptr selects the peer-memory scatter store
template <typename T>
static int launch_lines_rg(const void *src, void *dst, void *const *peer_host, int P, int N, int64_t line_stride,
                           int64_t n_inner, int64_t n_outer, int64_t outer_stride, int64_t outer_start, int inverse,
                           double scale, cudaStream_t s, int64_t d_total_override = 0) {
    typedef typename C2<T>::type C;
    {
        bool done = false;
        int rct = launch_lines_tma<T>(src, dst, peer_host, P, N, line_stride, n_inner, n_outer, outer_stride, outer_start,
                                      inverse, scale, s, d_total_override, &done);
        if (rct || done) return rct;
    }
    int dtype = sizeof(T) == 4 ? NBK_F4 : NBK_F8;
    void *tw;
    int rc = get_twiddle(N, dtype, s, &tw);
    if (rc) return rc;
    // tile width: 128-byte runs; the peer-memory scatter uses 256-byte runs (measured 17 % faster over NVLink; NBK_FFT_PEER_RUN=128 restores the narrow tile)
    static int peer_run = -1;
    if (peer_run < 0) {
        const char *e = getenv("NBK_FFT_PEER_RUN");
        peer_run = e ? atoi(e) : 256;
        if (peer_run != 128 && peer_run != 256) peer_run = 256;
    }
    int B = (peer_host ? peer_run : 128) / (int)sizeof(C);
    if (B > 16) B = 16;
    // experiment knobs: NBK_FFT_LINE_B (tile width), NBK_FFT_LINE_NT (threads per CTA: 128 / 256 / 512)
    static int knob_b = -1, knob_nt = -1;
    if (knob_b < 0) {
        const char *e = getenv("NBK_FFT_LINE_B");
        knob_b = e ? atoi(e) : 0;
        e = getenv("NBK_FFT_LINE_NT");
        knob_nt = e ? atoi(e) : 0;
    }
    if (!peer_host && (knob_b == 2 || knob_b == 4 || knob_b == 8 || knob_b == 16)) B = knob_b;
    while (B > 1 && ((size_t)N * (B + 2) * sizeof(C) > 220 * 1024 || B / 2 >= n_inner)) B >>= 1;
    size_t smem = (size_t)N * (B + 2) * sizeof(C);
    NBK_CHECK_ARG(smem <= 227 * 1024, "fft_lines: N=%d does not fit in shared memory", N);
    int64_t tiles_inner = (n_inner + B - 1) / B;
    int64_t n_tiles = tiles_inner * n_outer;
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    int nthreads = (per_sm == 1 && B >= 4) ? 512 : 256;
    if (!peer_host && knob_nt == 128 && B >= 2 && B <= 8) nthreads = 128;
    if (!peer_host && knob_nt == 512 && B >= 4) nthreads = 512;
    if (nthreads == 128 && per_sm > 4) per_sm = 4;
    if (nthreads == 256 && per_sm > 2) per_sm = 2;       // 128 registers per thread
    if (nthreads == 512) per_sm = 1;
    int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
    PeerPtrs<C> peers;
    for (int i = 0; i < NBK_MAX_PEERS; i++) peers.p[i] = (peer_host && i < P) ? (C *)peer_host[i] : nullptr;
    const int n_per = peer_host ? N / P : N;
    const int64_t d_total = d_total_override ? d_total_override : (peer_host ? n_outer * P : 0);
    static int prefetch = -1;
    if (prefetch < 0) {
        const char *e = getenv("NBK_FFT_PREFETCH");
        prefetch = (e && e[0] == '0') ? 0 : 1;
    }
    const int first_per_thread = (int)(((int64_t)(N >> 3) * B) / nthreads);
    const bool exact = ((int64_t)(N >> 3) * B) % nthreads == 0;
#define LAUNCH_RGP(BB, NTT, IT)                                                                                       \
        if (peer_host) {                                                                                           \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_rgp<T, BB, true, NTT, IT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_lines_rgp<T, BB, true, NTT, IT><<<(int)g, NTT, smem, s>>>((const C *)src, (C *)dst, peers, (const C *)tw, N, \
                ilog2(N), line_stride, n_inner, tiles_inner, n_tiles, outer_stride, n_per, d_total, outer_start, inverse, (T)scale); \
        } else {                                                                                                   \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_rgp<T, BB, false, NTT, IT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_lines_rgp<T, BB, false, NTT, IT><<<(int)g, NTT, smem, s>>>((const C *)src, (C *)dst, peers, (const C *)tw, N, \
                ilog2(N), line_stride, n_inner, tiles_inner, n_tiles, outer_stride, n_per, d_total, outer_start, inverse, (T)scale); \
        }
    // the common shapes: two first-stage butterflies per thread (512^3: B=8/16, 256 threads; 1024^3: B=8, 512 threads)
    if (prefetch && exact && first_per_thread == 2) {
        bool done = true;
        if (nthreads == 512 && B == 8) { LAUNCH_RGP(8, 512, 2) }
        else if (nthreads == 512 && B == 16) { LAUNCH_RGP(16, 512, 2) }
        else if (nthreads == 256 && B == 8) { LAUNCH_RGP(8, 256, 2) }
        else if (nthreads == 256 && B == 16) { LAUNCH_RGP(16, 256, 2) }
        else done = false;
        if (done) { NBK_LAUNCHED(); return NBK_OK; }
    }
#undef LAUNCH_RGP
#define LAUNCH_RG(BB, NTT)                                                                                            \
    case BB:                                                                                                       \
        if (peer_host) {                                                                                           \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_rg<T, BB, true, NTT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_lines_rg<T, BB, true, NTT><<<(int)g, NTT, smem, s>>>((const C *)src, (C *)dst, peers, (const C *)tw, N, \
                ilog2(N), line_stride, n_inner, tiles_inner, n_tiles, outer_stride, n_per, d_total, outer_start, inverse, (T)scale); \
        } else {                                                                                                   \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_rg<T, BB, false, NTT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_lines_rg<T, BB, false, NTT><<<(int)g, NTT, smem, s>>>((const C *)src, (C *)dst, peers, (const C *)tw, N, \
                ilog2(N), line_stride, n_inner, tiles_inner, n_tiles, outer_stride, n_per, d_total, outer_start, inverse, (T)scale); \
        }                                                                                                          \
        break;
    if (nthreads == 128) {
        switch (B) {
            LAUNCH_RG(2, 128) LAUNCH_RG(4, 128) LAUNCH_RG(8, 128)
            default: nbk_set_error("fft_lines: internal tile width %d", B); return NBK_ERR_ARG;
        }
    } else if (nthreads == 512) {
        switch (B) {
            LAUNCH_RG(4, 512) LAUNCH_RG(8, 512) LAUNCH_RG(16, 512)
            default: nbk_set_error("fft_lines: internal tile width %d", B); return NBK_ERR_ARG;
        }
    } else {
        switch (B) {
            LAUNCH_RG(1, 256) LAUNCH_RG(2, 256) LAUNCH_RG(4, 256) LAUNCH_RG(8, 256) LAUNCH_RG(16, 256)
            default: nbk_set_error("fft_lines: internal tile width %d", B); return NBK_ERR_ARG;
        }
    }
#undef LAUNCH_RG
    NBK_LAUNCHED();
    return NBK_OK;
}

template <typename T>
static int launch_lines(const void *data, void *dst, int N, int64_t line_stride, int64_t n_inner, int64_t n_outer,
                        int64_t outer_stride, int inverse, double scale, cudaStream_t s) {
    typedef typename C2<T>::type C;
    int dtype = sizeof(T) == 4 ? NBK_F4 : NBK_F8;
    if (N == 1) {
        if (scale != 1.0 || dst != data) {
            nbk_set_error("fft_lines: N == 1 with scale / out of place is not supported");
            return NBK_ERR_UNSUPPORTED;
        }
        return NBK_OK;
    }
    if (use_reg_lines(N))
        return launch_lines_rg<T>(data, dst, nullptr, 1, N, line_stride, n_inner, n_outer, outer_stride, 0, inverse, scale, s);
    void *tw;
    int rc = get_twiddle(N, dtype, s, &tw);
    if (rc) return rc;
    // two tile buffers [N][B+1] + twiddle table [N].  B * sizeof(C) = 128 bytes makes every quarter-warp shared
    // access one full padded row (bank-conflict free for any row), so keep that width as long as it fits and run
    // one 512-thread CTA per SM; narrower tiles only for very long lines.
    int B = 128 / (int)sizeof(C);
    while (B > 1 && ((size_t)N * (2 * (B + 1) + 1) * sizeof(C) > 220 * 1024 || B / 2 >= n_inner)) B >>= 1;
    size_t smem = (size_t)N * (2 * (B + 1) + 1) * sizeof(C);
    NBK_CHECK_ARG(smem <= 227 * 1024, "fft_lines: N=%d does not fit in shared memory", N);
    int64_t tiles_inner = (n_inner + B - 1) / B;
    int64_t n_tiles = tiles_inner * n_outer;
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
    const int nthreads = (per_sm == 1 && (int64_t)N * B >= 4096) ? 512 : 256;
#define LAUNCH_LINES(BB)                                                                                          \
    case BB:                                                                                                      \
        NBK_CUDA(cudaFuncSetAttribute(k_fft_lines<T, BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_fft_lines<T, BB><<<(int)g, nthreads, smem, s>>>((const C *)data, (C *)dst, (const C *)tw, N, ilog2(N), line_stride, n_inner, \
                                                     tiles_inner, n_tiles, outer_stride, inverse, (T)scale);      \
        break;
    switch (B) {
        LAUNCH_LINES(1) LAUNCH_LINES(2) LAUNCH_LINES(4) LAUNCH_LINES(8) LAUNCH_LINES(16)
        default: nbk_set_error("fft_lines: internal tile width %d", B); return NBK_ERR_ARG;
    }
#undef LAUNCH_LINES
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fft_lines(void *cplx, int dtype, int64_t n_line, int64_t line_stride, int64_t n_inner,
                             int64_t n_outer, int64_t outer_stride, int inverse, double scale, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_lines: bad dtype %d", dtype);
    NBK_CHECK_ARG(is_pow2(n_line) && n_line <= 8192, "fft_lines: line length %lld is not a supported power of two",
                  (long long)n_line);
    if (n_inner <= 0 || n_outer <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_lines<float>(cplx, cplx, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
    return launch_lines<double>(cplx, cplx, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
}

// out-of-place variant (same layout for src and dst)
extern "C" int nbk_fft_lines_oop(const void *src, void *dst, int dtype, int64_t n_line, int64_t line_stride,
                                 int64_t n_inner, int64_t n_outer, int64_t outer_stride, int inverse, double scale,
                                 void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_lines_oop: bad dtype %d", dtype);
    NBK_CHECK_ARG(is_pow2(n_line) && n_line >= 2 && n_line <= 8192, "fft_lines_oop: line length %lld unsupported", (long long)n_line);
    if (n_inner <= 0 || n_outer <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_lines<float>(src, dst, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
    return launch_lines<double>(src, dst, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
}

template <typename T>
static int launch_lines_scatter(const void *src, void *const *peer_host, int N, int64_t n_inner, int64_t n_outer,
                                int64_t outer_start, int P, int inverse, double scale, cudaStream_t s,
                                int64_t d_total_override = 0) {
    if (use_reg_lines(N))
        return launch_lines_rg<T>(src, nullptr, peer_host, P, N, n_inner, n_inner, n_outer, (int64_t)N * n_inner, outer_start,
                                  inverse, scale, s, d_total_override);
    typedef typename C2<T>::type C;
    int dtype = sizeof(T) == 4 ? NBK_F4 : NBK_F8;
    void *tw;
    int rc = get_twiddle(N, dtype, s, &tw);
    if (rc) return rc;
    int B = pick_B(N, (int)sizeof(C), n_inner);
    size_t smem = (size_t)N * (B + 2) * sizeof(C);
    NBK_CHECK_ARG(smem <= 227 * 1024, "fft_lines_scatter: N=%d does not fit in shared memory", N);
    int64_t tiles_inner = (n_inner + B - 1) / B;
    int64_t n_tiles = tiles_inner * n_outer;
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
    PeerPtrs<C> peers;
    for (int i = 0; i < NBK_MAX_PEERS; i++) peers.p[i] = i < P ? (C *)peer_host[i] : nullptr;
#define LAUNCH_LS(BB)                                                                                                \
    case BB:                                                                                                         \
        NBK_CUDA(cudaFuncSetAttribute(k_fft_lines_scatter<T, BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        k_fft_lines_scatter<T, BB><<<(int)g, 256, smem, s>>>((const C *)src, peers, (const C *)tw, N, ilog2(N), n_inner, \
                                                             tiles_inner, n_tiles, N / P,                              \
                                                             d_total_override ? d_total_override : n_outer * P, outer_start, \
                                                             inverse, (T)scale);                                     \
        break;
    switch (B) {
        LAUNCH_LS(1) LAUNCH_LS(2) LAUNCH_LS(4) LAUNCH_LS(8) LAUNCH_LS(16)
        default: nbk_set_error("fft_lines_scatter: internal tile width %d", B); return NBK_ERR_ARG;
    }
#undef LAUNCH_LS
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fft_lines_scatter(const void *src, void *const *peer_ptrs_host, int dtype, int64_t n_line,
                                     int64_t n_inner, int64_t n_outer, int64_t outer_start, int P, int inverse,
                                     double scale, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_lines_scatter: bad dtype %d", dtype);
    NBK_CHECK_ARG(is_pow2(n_line) && n_line >= 2 && n_line <= 8192, "fft_lines_scatter: line length %lld unsupported", (long long)n_line);
    NBK_CHECK_ARG(P >= 1 && P <= NBK_MAX_PEERS && n_line % P == 0, "fft_lines_scatter: bad peer count %d", P);
    if (n_inner <= 0 || n_outer <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_lines_scatter<float>(src, peer_ptrs_host, (int)n_line, n_inner, n_outer, outer_start, P, inverse, scale, s);
    return launch_lines_scatter<double>(src, peer_ptrs_host, (int)n_line, n_inner, n_outer, outer_start, P, inverse, scale, s);
}

template <typename T>
static int launch_z(const void *in, void *out, int64_t rows, int Nz, bool forward, double scale, cudaStream_t s) {
    typedef typename C2<T>::type C;
    int dtype = sizeof(T) == 4 ? NBK_F4 : NBK_F8;
    int M = Nz / 2;
    void *twM, *twN;
    int rc = get_twiddle(M, dtype, s, &twM);
    if (rc) return rc;
    rc = get_twiddle(Nz, dtype, s, &twN);
    if (rc) return rc;
    if (forward && lines_mode() == 2 && (M == 128 || M == 256 || M == 512) && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
        ((size_t)Nz * sizeof(T)) % 16 == 0) {
        // warp-per-row TMA pass: 12 warps, per-warp ring of row buffers filling the SM's shared memory
        constexpr int NWZ = 12;
        const size_t rowb = (size_t)M * sizeof(C);
        const size_t twb = ((size_t)Nz + 7 * (M / 8) + 56) * sizeof(C);       // W_N | stage-1 table | stage-2 table
        int nbuf = (int)(((size_t)224 * 1024 - twb - 1024) / (NWZ * rowb));
        if (nbuf > 4) nbuf = 4;
        if (nbuf < 2) nbuf = 2;
        static int knob_nb = -1;
        if (knob_nb < 0) { const char *e = getenv("NBK_FFT_Z_NBUF"); knob_nb = e ? atoi(e) : 0; }
        if (knob_nb >= 1 && knob_nb <= nbuf) nbuf = knob_nb;
        const size_t smem = twb + (size_t)NWZ * nbuf * rowb + (size_t)NWZ * nbuf * 8 + 128;
        NBK_CHECK_ARG(smem <= 227 * 1024, "fft z pass: Nz=%d does not fit in shared memory", Nz);
        int64_t g = (rows + NWZ - 1) / NWZ;
        if (g > NBK_SM_COUNT) g = NBK_SM_COUNT;
#define LAUNCH_ZT(LMM)                                                                                            \
        do {                                                                                                      \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_z_r2c_tma<T, LMM, NWZ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_z_r2c_tma<T, LMM, NWZ><<<(int)g, 32 * NWZ, smem, s>>>((const T *)in, (C *)out, (const C *)twN, rows, (T)scale, nbuf); \
        } while (0)
        if (M == 512) LAUNCH_ZT(9); else if (M == 256) LAUNCH_ZT(8); else LAUNCH_ZT(7);
#undef LAUNCH_ZT
        NBK_LAUNCHED();
        return NBK_OK;
    }
    if (forward && M >= 64 && M <= 256 * (sizeof(T) == 4 ? 16 : 8) && use_reg_lines(M)) {   // the tile must fit the registers
        // register-I/O variant: 256 threads hold the whole tile across the last stage (M * B <= 256 V)
        const int V = sizeof(T) == 4 ? 16 : 8;
        int B = 16;
        while (B > 1 && (M * B > 256 * V || B / 2 >= rows)) B >>= 1;
        size_t smem = ((size_t)M * (B + 1) + Nz + 7 * (M / 8)) * sizeof(C);   // tile | W_N | first-stage twiddles
        NBK_CHECK_ARG(smem <= 227 * 1024, "fft z pass: Nz=%d does not fit in shared memory", Nz);
        int64_t n_tiles = (rows + B - 1) / B;
        int per_sm = (int)((227 * 1024) / (smem + 1024));
        if (per_sm < 1) per_sm = 1;
        if (per_sm > 4) per_sm = 4;
        int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
#define LAUNCH_ZRG(BB)                                                                                            \
    case BB: {                                                                                                    \
        NBK_CUDA(cudaFuncSetAttribute(k_fft_z_r2c_rg<T, BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        int occ = 1;   /* persistent tile loop: exactly one wave of resident CTAs (registers, not shared memory, limit it) */ \
        NBK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_fft_z_r2c_rg<T, BB>, 256, smem));           \
        if (occ < 1) occ = 1;                                                                                     \
        if (g > (int64_t)NBK_SM_COUNT * occ) g = (int64_t)NBK_SM_COUNT * occ;                                      \
        k_fft_z_r2c_rg<T, BB><<<(int)g, 256, smem, s>>>((const T *)in, (C *)out, (const C *)twN, Nz, ilog2(M), rows, (T)scale); \
        break; }
        switch (B) {
            LAUNCH_ZRG(1) LAUNCH_ZRG(2) LAUNCH_ZRG(4) LAUNCH_ZRG(8) LAUNCH_ZRG(16)
            default: nbk_set_error("fft z pass: internal tile width %d", B); return NBK_ERR_ARG;
        }
#undef LAUNCH_ZRG
        NBK_LAUNCHED();
        return NBK_OK;
    }
    int B = pick_B(M, (int)sizeof(C), rows);
    size_t smem = ((size_t)M * (B + 2) + 8) * sizeof(C);     // tile [M][B+1] (+8 skew) + twiddle table [M]
    NBK_CHECK_ARG(smem <= 227 * 1024, "fft z pass: Nz=%d does not fit in shared memory", Nz);
    int64_t n_tiles = (rows + B - 1) / B;
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int64_t g = n_tiles < (int64_t)NBK_SM_COUNT * per_sm ? n_tiles : (int64_t)NBK_SM_COUNT * per_sm;
#define LAUNCH_Z(BB)                                                                                              \
    case BB:                                                                                                      \
        if (forward) {                                                                                            \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_z_r2c<T, BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_z_r2c<T, BB><<<(int)g, 256, smem, s>>>((const T *)in, (C *)out, (const C *)twM, (const C *)twN, Nz, \
                                                         ilog2(M), rows, (T)scale);                               \
        } else {                                                                                                  \
            NBK_CUDA(cudaFuncSetAttribute(k_fft_z_c2r<T, BB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
            k_fft_z_c2r<T, BB><<<(int)g, 256, smem, s>>>((const C *)in, (T *)out, (const C *)twM, (const C *)twN, Nz, \
                                                         ilog2(M), rows);                                         \
        }                                                                                                         \
        break;
    switch (B) {
        LAUNCH_Z(1) LAUNCH_Z(2) LAUNCH_Z(4) LAUNCH_Z(8) LAUNCH_Z(16)
        default: nbk_set_error("fft z pass: internal tile width %d", B); return NBK_ERR_ARG;
    }
#undef LAUNCH_Z
    NBK_LAUNCHED();
    return NBK_OK;
}

static int check_dims(const char *who, int dtype, int64_t Nx, int64_t Ny, int64_t Nz) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "%s: bad dtype %d", who, dtype);
    NBK_CHECK_ARG(is_pow2(Nx) && is_pow2(Ny) && is_pow2(Nz) && Nz >= 4 && Nx <= 8192 && Ny <= 8192 && Nz <= 16384,
                  "%s: Nmesh (%lld,%lld,%lld) unsupported: each side must be a power of two (Nz >= 4)", who,
                  (long long)Nx, (long long)Ny, (long long)Nz);
    return NBK_OK;
}

// z pass alone: real rows [rows][Nz] -> complex rows [rows][Nz/2+1]
extern "C" int nbk_fft_z_forward(const void *real, void *cplx, int dtype, int64_t rows, int64_t Nz, void *stream) {
    int rc = check_dims("fft_z_forward", dtype, 1, 1, Nz);
    if (rc) return rc;
    if (rows <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    return (dtype == NBK_F4) ? launch_z<float>(real, cplx, rows, (int)Nz, true, 1.0, s)
                             : launch_z<double>(real, cplx, rows, (int)Nz, true, 1.0, s);
}

extern "C" int nbk_fft_zy_forward(const void *real, void *cplx, int dtype, int64_t x_n, int64_t Ny, int64_t Nz,
                                  void *stream) {
    int rc = check_dims("fft_zy_forward", dtype, 1, Ny, Nz);
    if (rc) return rc;
    if (x_n <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t Nzc = Nz / 2 + 1;
    rc = (dtype == NBK_F4) ? launch_z<float>(real, cplx, x_n * Ny, (int)Nz, true, 1.0, s)
                           : launch_z<double>(real, cplx, x_n * Ny, (int)Nz, true, 1.0, s);
    if (rc) return rc;
    return nbk_fft_lines(cplx, dtype, Ny, Nzc, Nzc, x_n, Ny * Nzc, 0, 1.0, stream);
}

extern "C" int nbk_fft_zy_backward(void *cplx, void *real, int dtype, int64_t x_n, int64_t Ny, int64_t Nz,
                                   void *stream) {
    int rc = check_dims("fft_zy_backward", dtype, 1, Ny, Nz);
    if (rc) return rc;
    if (x_n <= 0) return NBK_OK;
    cudaStream_t s = (cudaStream_t)stream;
    int64_t Nzc = Nz / 2 + 1;
    rc = nbk_fft_lines(cplx, dtype, Ny, Nzc, Nzc, x_n, Ny * Nzc, 1, 1.0, stream);
    if (rc) return rc;
    return (dtype == NBK_F4) ? launch_z<float>(cplx, real, x_n * Ny, (int)Nz, false, 1.0, s)
                             : launch_z<double>(cplx, real, x_n * Ny, (int)Nz, false, 1.0, s);
}

extern "C" int nbk_r2c(const void *real, void *cplx, int dtype, const int64_t *nmesh, double extra_scale, void *stream) {
    int rc = check_dims("r2c", dtype, nmesh[0], nmesh[1], nmesh[2]);
    if (rc) return rc;
    int64_t Nx = nmesh[0], Ny = nmesh[1], Nz = nmesh[2], Nzc = Nz / 2 + 1;
    rc = nbk_fft_zy_forward(real, cplx, dtype, Nx, Ny, Nz, stream);
    if (rc) return rc;
    double scale = extra_scale / ((double)Nx * (double)Ny * (double)Nz);
    if (Nx == 1) return nbk_scale(cplx, dtype, 2 * Ny * Nzc, scale, stream);
    return nbk_fft_lines(cplx, dtype, Nx, Ny * Nzc, Ny * Nzc, 1, 0, 0, scale, stream);
}

// c2r destroys its complex input unless `work` (same size as cplx) is given
extern "C" int nbk_c2r(const void *cplx, void *real, int dtype, const int64_t *nmesh, void *work, void *stream) {
    int rc = check_dims("c2r", dtype, nmesh[0], nmesh[1], nmesh[2]);
    if (rc) return rc;
    int64_t Nx = nmesh[0], Ny = nmesh[1], Nz = nmesh[2], Nzc = Nz / 2 + 1;
    void *c = const_cast<void *>(cplx);
    if (work && work != cplx) {
        size_t bytes = (size_t)Nx * Ny * Nzc * (dtype == NBK_F4 ? 8 : 16);
        NBK_CUDA(cudaMemcpyAsync(work, cplx, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        c = work;
    }
    rc = nbk_fft_lines(c, dtype, Nx, Ny * Nzc, Ny * Nzc, 1, 0, 1, 1.0, stream);
    if (rc) return rc;
    return nbk_fft_zy_backward(c, real, dtype, Nx, Ny, Nz, stream);
}

// ---------------------------------------------------------------------------------------------
// slab <-> pencil transposes for P > 1 (row copies of Nzc complex, coalesced along kz)
// ---------------------------------------------------------------------------------------------
// generic: dst[(a*nb + b)*row + k] = src[(b*na + a)*row + k] with an extra block split described by the callers
template <typename C>
__global__ void __launch_bounds__(256)
k_row_permute(const C *__restrict__ src, C *__restrict__ dst, int64_t n_rows, int row, int64_t d0, int64_t d1,
              int64_t d2, int64_t s0, int64_t s1, int64_t s2) {
    // destination row index r = (i0*d1 + i1)*d2 + i2  ->  source row = i0*s0 + i1*s1 + i2*s2
    int lanes_per_row = 32;
    int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / lanes_per_row;
    int lane = threadIdx.x % lanes_per_row;
    int64_t nw = ((int64_t)gridDim.x * blockDim.x) / lanes_per_row;
    for (int64_t r = wid; r < n_rows; r += nw) {
        int64_t i2 = r % d2;
        int64_t i1 = (r / d2) % d1;
        int64_t i0 = r / (d2 * d1);
        const C *sp = src + (i0 * s0 + i1 * s1 + i2 * s2) * row;
        C *dp = dst + r * row;
        for (int k = lane; k < row; k += lanes_per_row) dp[k] = sp[k];
    }
}

template <typename C>
static int launch_permute(const void *src, void *dst, int64_t d0, int64_t d1, int64_t d2, int64_t s0, int64_t s1,
                          int64_t s2, int row, cudaStream_t s) {
    int64_t n_rows = d0 * d1 * d2;
    if (n_rows == 0) return NBK_OK;
    int g = nbk_grid_for(n_rows * 32, 256, 8);
    k_row_permute<C><<<g, 256, 0, s>>>((const C *)src, (C *)dst, n_rows, row, d0, d1, d2, s0, s1, s2);
    NBK_LAUNCHED();
    return NBK_OK;
}

#define PERMUTE(dtype, ...)                                                          \
    ((dtype) == NBK_F4 ? launch_permute<float2>(__VA_ARGS__) : launch_permute<double2>(__VA_ARGS__))

// [x_n][Ny][Nzc] -> [P][y_n][x_n][Nzc]   (dst rows (p, yl, x) <- src row (x, p*y_n + yl))
extern "C" int nbk_transpose_pack(const void *src, void *dst, int dtype, int64_t x_n, int64_t Ny, int64_t Nzc,
                                  int64_t P, void *stream) {
    NBK_CHECK_ARG(P > 0 && Ny % P == 0, "transpose_pack: Ny %% P != 0");
    int64_t y_n = Ny / P;
    // dst index (i0=p, i1=yl, i2=x): src row = x*Ny + p*y_n + yl
    return PERMUTE(dtype, src, dst, P, y_n, x_n, y_n, 1, Ny, (int)Nzc, (cudaStream_t)stream);
}
// [P][y_n][x_n][Nzc] (block q came from rank q) -> [y_n][Nx][Nzc], Nx = P*x_n
extern "C" int nbk_transpose_unpack(const void *src, void *dst, int dtype, int64_t y_n, int64_t Nx, int64_t Nzc,
                                    int64_t P, void *stream) {
    NBK_CHECK_ARG(P > 0 && Nx % P == 0, "transpose_unpack: Nx %% P != 0");
    int64_t x_n = Nx / P;
    // dst (i0=yl, i1=q, i2=xl): src row = (q*y_n + yl)*x_n + xl
    return PERMUTE(dtype, src, dst, y_n, P, x_n, x_n, y_n * x_n, 1, (int)Nzc, (cudaStream_t)stream);
}
// inverse of unpack: [y_n][Nx][Nzc] -> [P][y_n][x_n][Nzc]
extern "C" int nbk_transpose_pack_back(const void *src, void *dst, int dtype, int64_t y_n, int64_t Nx, int64_t Nzc,
                                       int64_t P, void *stream) {
    NBK_CHECK_ARG(P > 0 && Nx % P == 0, "transpose_pack_back: Nx %% P != 0");
    int64_t x_n = Nx / P;
    // dst (i0=q, i1=yl, i2=xl): src row = yl*Nx + q*x_n + xl
    return PERMUTE(dtype, src, dst, P, y_n, x_n, x_n, Nx, 1, (int)Nzc, (cudaStream_t)stream);
}
// inverse of pack: [P][y_n][x_n][Nzc] -> [x_n][Ny][Nzc]
extern "C" int nbk_transpose_unpack_back(const void *src, void *dst, int dtype, int64_t x_n, int64_t Ny, int64_t Nzc,
                                         int64_t P, void *stream) {
    NBK_CHECK_ARG(P > 0 && Ny % P == 0, "transpose_unpack_back: Ny %% P != 0");
    int64_t y_n = Ny / P;
    // dst (i0=x, i1=p, i2=yl): src row = (p*y_n + yl)*x_n + x
    return PERMUTE(dtype, src, dst, x_n, P, y_n, 1, y_n * x_n, x_n, (int)Nzc, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Complex-dtype meshes (ParticleMesh(dtype='c16'/'c8'): pmesh then runs c2c transforms and keeps all N^3 modes,
// `ComplexField.compressed == False`, fftpower.py:572; convpower/catalog.py:151-176).  On this path the
// configuration-space field is real-valued, so its full spectrum is the Hermitian completion of the r2c result:
//   full[ix][iy][iz] = comp[ix][iy][iz]                                   iz <= Nz/2
//                    = conj(comp[(-ix) % Nx][(-iy) % Ny][Nz - iz])        iz >  Nz/2
// One read of the compressed field, one write of the full one (a c2c transform would move three times as much).
// ---------------------------------------------------------------------------------------------
template <typename C>
__global__ void __launch_bounds__(256)
k_hermitian_expand(const C *__restrict__ comp, C *__restrict__ full, int Nx, int Ny, int Nz) {
    const int Nzc = Nz / 2 + 1;
    const int64_t rows = (int64_t)Nx * Ny;
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = w0; row < rows; row += nw) {
        const int ix = (int)(row / Ny), iy = (int)(row - (int64_t)ix * Ny);
        const int mx = ix ? Nx - ix : 0, my = iy ? Ny - iy : 0;
        const C *a = comp + row * Nzc;
        const C *b = comp + ((int64_t)mx * Ny + my) * Nzc;
        C *o = full + row * Nz;
        for (int iz = lane; iz < Nz; iz += 32) {
            C v;
            if (iz < Nzc) v = a[iz];
            else { v = b[Nz - iz]; v.y = -v.y; }
            o[iz] = v;
        }
    }
}

template <typename C>
__global__ void __launch_bounds__(256)
k_hermitian_compress(const C *__restrict__ full, C *__restrict__ comp, int64_t rows, int Nz) {
    const int Nzc = Nz / 2 + 1;
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = w0; row < rows; row += nw)
        for (int iz = lane; iz < Nzc; iz += 32) comp[row * Nzc + iz] = full[row * Nz + iz];
}

extern "C" int nbk_hermitian_expand(const void *comp, void *full, int dtype, const int64_t *nmesh, void *stream) {
    // power-of-two sides (the transform of nbk_r2c) or the even 7-smooth sides of the mixed-radix nbk_r2c_mr
    int rc = (is_pow2(nmesh[0]) && is_pow2(nmesh[1]) && is_pow2(nmesh[2]))
                 ? check_dims("hermitian_expand", dtype, nmesh[0], nmesh[1], nmesh[2])
                 : nbk_check_mixed_dims("hermitian_expand", dtype, nmesh[0], nmesh[1], nmesh[2]);
    if (rc) return rc;
    NBK_CHECK_ARG(comp != nullptr && full != nullptr && comp != full, "hermitian_expand: needs two distinct buffers");
    int64_t rows = nmesh[0] * nmesh[1];
    int g = nbk_grid_for(rows * 32, 256, 8);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4) k_hermitian_expand<float2><<<g, 256, 0, s>>>((const float2 *)comp, (float2 *)full, (int)nmesh[0], (int)nmesh[1], (int)nmesh[2]);
    else k_hermitian_expand<double2><<<g, 256, 0, s>>>((const double2 *)comp, (double2 *)full, (int)nmesh[0], (int)nmesh[1], (int)nmesh[2]);
    NBK_LAUNCHED();
    return NBK_OK;
}

// the stored half of a full spectrum (the inverse of nbk_hermitian_expand for Hermitian fields; rows = Nx * Ny of this rank)
extern "C" int nbk_hermitian_compress(const void *full, void *comp, int dtype, int64_t rows, int64_t Nz, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "hermitian_compress: bad dtype %d", dtype);
    NBK_CHECK_ARG(rows >= 0 && Nz >= 2 && comp != full, "hermitian_compress: bad arguments");
    if (rows == 0) return NBK_OK;
    int g = nbk_grid_for(rows * 32, 256, 8);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4) k_hermitian_compress<float2><<<g, 256, 0, s>>>((const float2 *)full, (float2 *)comp, rows, (int)Nz);
    else k_hermitian_compress<double2><<<g, 256, 0, s>>>((const double2 *)full, (double2 *)comp, rows, (int)Nz);
    NBK_LAUNCHED();
    return NBK_OK;
}

// ---------------------------------------------------------------------------------------------
// Fourier-space resampling to another mesh size (pmesh `Field.resample`, called from base/mesh.py:317-327 when
// compute(Nmesh=...) asks for a size other than the source's): the modes both meshes represent are copied, the rest
// of the destination is zero (down-sampling = truncation, up-sampling = zero padding; the normalised transform keeps
// amplitudes, so the mean is preserved).  Per axis a destination index maps to the source index with the same integer
// frequency label, labels in [-Nmin/2, Nmin/2) (Nyquist negative, meshtools.py:150-153); along the Hermitian-compressed
// axis indices 0 .. Nmin/2 map to themselves.  Single GPU, compressed layout [Nx][Ny][Nz/2+1].
// ---------------------------------------------------------------------------------------------
template <typename C>
__global__ void __launch_bounds__(256)
k_resample_complex(const C *__restrict__ src, C *__restrict__ dst, int sx, int sy, int sz, int dx, int dy, int dz) {
    const int szc = sz / 2 + 1, dzc = dz / 2 + 1;
    const int mzc = (sz < dz ? sz : dz) / 2 + 1;
    const int64_t rows = (int64_t)dx * dy;
    const int lane = threadIdx.x & 31;
    const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = w0; row < rows; row += nw) {
        const int ix = (int)(row / dy), iy = (int)(row - (int64_t)ix * dy);
        const int jx = nbk_freq(ix, dx), jy = nbk_freq(iy, dy);
        const int mx = sx < dx ? sx : dx, my = sy < dy ? sy : dy;
        const bool ok = 2 * jx >= -mx && 2 * jx < mx && 2 * jy >= -my && 2 * jy < my;
        const C *s = src + ((int64_t)(jx < 0 ? jx + sx : jx) * sy + (jy < 0 ? jy + sy : jy)) * szc;
        C *d = dst + row * dzc;
        for (int iz = lane; iz < dzc; iz += 32) d[iz] = (ok && iz < mzc) ? s[iz] : C{0, 0};
    }
}

extern "C" int nbk_resample_complex(const void *src, void *dst, int dtype, const int64_t *nmesh_src,
                                    const int64_t *nmesh_dst, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "resample_complex: bad dtype %d", dtype);
    NBK_CHECK_ARG(src != nullptr && dst != nullptr && src != dst, "resample_complex: needs two distinct buffers");
    for (int d = 0; d < 3; d++)
        NBK_CHECK_ARG(nmesh_src[d] >= 2 && nmesh_dst[d] >= 2 && nmesh_src[d] < (1 << 24) && nmesh_dst[d] < (1 << 24) &&
                      nmesh_src[d] % 2 == 0 && nmesh_dst[d] % 2 == 0, "resample_complex: mesh sides must be even");
    int64_t rows = nmesh_dst[0] * nmesh_dst[1];
    int g = nbk_grid_for(rows * 32, 256, 8);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        k_resample_complex<float2><<<g, 256, 0, s>>>((const float2 *)src, (float2 *)dst, (int)nmesh_src[0], (int)nmesh_src[1],
                                                     (int)nmesh_src[2], (int)nmesh_dst[0], (int)nmesh_dst[1], (int)nmesh_dst[2]);
    else
        k_resample_complex<double2><<<g, 256, 0, s>>>((const double2 *)src, (double2 *)dst, (int)nmesh_src[0], (int)nmesh_src[1],
                                                      (int)nmesh_src[2], (int)nmesh_dst[0], (int)nmesh_dst[1], (int)nmesh_dst[2]);
    NBK_LAUNCHED();
    return NBK_OK;
}

// ---------------------------------------------------------------------------------------------
// Slab transpose as "line pass into send blocks" + bulk peer copies (P > 1).  The line pass (y pass of r2c, inverse x
// pass of c2r) stores its output rows directly in transposed order into P contiguous LOCAL blocks
//     send[p][kl][outer][inner]      kl = k % (N/P) the line frequency inside rank p's share, outer < n_outer
// and nbk_slab_push() moves block p into rank p's field [N/P][n_outer * P][n_inner] with one strided bulk copy per
// peer: rows of n_outer * n_inner contiguous elements (1 MB at 1024^3 on 8 GPUs) travel over NVLink on the copy
// engines at link rate, instead of the 128..256-byte remote stores of nbk_fft_lines_scatter.
// ---------------------------------------------------------------------------------------------
extern "C" int nbk_fft_lines_pack(const void *src, void *send, int dtype, int64_t n_line, int64_t n_inner, int64_t n_outer,
                                  int P, int inverse, double scale, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_lines_pack: bad dtype %d", dtype);
    NBK_CHECK_ARG(is_pow2(n_line) && n_line >= 2 && n_line <= 8192, "fft_lines_pack: line length %lld unsupported", (long long)n_line);
    NBK_CHECK_ARG(P >= 1 && P <= NBK_MAX_PEERS && n_line % P == 0, "fft_lines_pack: bad peer count %d", P);
    if (n_inner <= 0 || n_outer <= 0) return NBK_OK;
    const size_t cs = dtype == NBK_F4 ? 8 : 16;
    const size_t block = (size_t)(n_line / P) * n_outer * n_inner * cs;
    void *blocks[NBK_MAX_PEERS];
    for (int p = 0; p < P; p++) blocks[p] = (char *)send + (size_t)p * block;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_lines_scatter<float>(src, blocks, (int)n_line, n_inner, n_outer, 0, P, inverse, scale, s, n_outer);
    return launch_lines_scatter<double>(src, blocks, (int)n_line, n_inner, n_outer, 0, P, inverse, scale, s, n_outer);
}

// the same line pass restricted to the outer sub-range [o0, o0 + o_cnt) of the slab (the send blocks keep their full
// [kl][n_outer][inner] shape): lets the caller push one part of the slab while the next part is still being transformed
extern "C" int nbk_fft_lines_pack_range(const void *src, void *send, int dtype, int64_t n_line, int64_t n_inner,
                                        int64_t n_outer, int64_t o0, int64_t o_cnt, int P, int inverse, double scale,
                                        void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_lines_pack_range: bad dtype %d", dtype);
    NBK_CHECK_ARG(is_pow2(n_line) && n_line >= 2 && n_line <= 8192, "fft_lines_pack_range: line length %lld unsupported", (long long)n_line);
    NBK_CHECK_ARG(P >= 1 && P <= NBK_MAX_PEERS && n_line % P == 0, "fft_lines_pack_range: bad peer count %d", P);
    NBK_CHECK_ARG(o0 >= 0 && o_cnt >= 0 && o0 + o_cnt <= n_outer, "fft_lines_pack_range: bad sub-range");
    if (n_inner <= 0 || o_cnt <= 0) return NBK_OK;
    const size_t cs = dtype == NBK_F4 ? 8 : 16;
    const size_t block = (size_t)(n_line / P) * n_outer * n_inner * cs;
    void *blocks[NBK_MAX_PEERS];
    for (int p = 0; p < P; p++) blocks[p] = (char *)send + (size_t)p * block;
    const char *sub = (const char *)src + (size_t)o0 * n_line * n_inner * cs;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_lines_scatter<float>(sub, blocks, (int)n_line, n_inner, o_cnt, o0, P, inverse, scale, s, n_outer);
    return launch_lines_scatter<double>(sub, blocks, (int)n_line, n_inner, o_cnt, o0, P, inverse, scale, s, n_outer);
}

// nbk_slab_push for the outer sub-range [o0, o0 + o_cnt) of every row
extern "C" int nbk_slab_push_range(const void *send, void *const *peer_ptrs_host, int dtype, int64_t rows_per_peer,
                                   int64_t n_outer, int64_t n_inner, int64_t outer_start, int64_t o0, int64_t o_cnt, int P,
                                   int rank, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "slab_push_range: bad dtype %d", dtype);
    NBK_CHECK_ARG(P >= 1 && P <= NBK_MAX_PEERS && rank >= 0 && rank < P, "slab_push_range: bad peer count / rank");
    NBK_CHECK_ARG(o0 >= 0 && o_cnt >= 0 && o0 + o_cnt <= n_outer, "slab_push_range: bad sub-range");
    if (rows_per_peer <= 0 || o_cnt <= 0 || n_inner <= 0) return NBK_OK;
    const size_t cs = dtype == NBK_F4 ? 8 : 16;
    const size_t spitch = (size_t)n_outer * n_inner * cs;           // one kl row of my block
    const size_t dpitch = spitch * P;                               // the same row of the destination field
    const size_t width = (size_t)o_cnt * n_inner * cs;
    cudaStream_t s = (cudaStream_t)stream;
    for (int i = 0; i < P; i++) {
        const int p = (rank + i) % P;                               // every rank starts with a different peer
        const char *srcp = (const char *)send + (size_t)p * rows_per_peer * spitch + (size_t)o0 * n_inner * cs;
        char *dstp = (char *)peer_ptrs_host[p] + (size_t)(outer_start + o0) * n_inner * cs;
        NBK_CUDA(cudaMemcpy2DAsync(dstp, dpitch, srcp, spitch, width, (size_t)rows_per_peer, cudaMemcpyDeviceToDevice, s));
    }
    return NBK_OK;
}

extern "C" int nbk_slab_push(const void *send, void *const *peer_ptrs_host, int dtype, int64_t rows_per_peer,
                             int64_t n_outer, int64_t n_inner, int64_t outer_start, int P, int rank, void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "slab_push: bad dtype %d", dtype);
    NBK_CHECK_ARG(P >= 1 && P <= NBK_MAX_PEERS && rank >= 0 && rank < P, "slab_push: bad peer count / rank");
    if (rows_per_peer <= 0 || n_outer <= 0 || n_inner <= 0) return NBK_OK;
    const size_t cs = dtype == NBK_F4 ? 8 : 16;
    const size_t width = (size_t)n_outer * n_inner * cs;            // one kl row of my block
    const size_t dpitch = width * P;                                // the same row of the destination field
    cudaStream_t s = (cudaStream_t)stream;
    for (int i = 0; i < P; i++) {
        const int p = (rank + i) % P;                               // every rank starts with a different peer
        const char *srcp = (const char *)send + (size_t)p * rows_per_peer * width;
        char *dstp = (char *)peer_ptrs_host[p] + (size_t)outer_start * n_inner * cs;
        NBK_CUDA(cudaMemcpy2DAsync(dstp, dpitch, srcp, width, width, (size_t)rows_per_peer, cudaMemcpyDeviceToDevice, s));
    }
    return NBK_OK;
}
