// Mixed-radix 3-D real<->complex FFT for mesh sides N = 2^a 3^b 5^c 7^d (RealField.r2c / ComplexField.c2r on meshes such
// as 384, 768, 1000 or 1536 per side; base/mesh.py:228,237).  Same layout, normalisation and precision contract as the
// power-of-two transform of fft.cu, which keeps serving every power-of-two mesh: forward scaled by 1/prod(N) (times the
// caller's scale), backward unnormalised, last axis Hermitian-compressed to Nz/2+1.
//
// One kernel family, one CTA per tile of B side-by-side lines held whole in shared memory ([N][B+1] padded rows; the B
// adjacent columns are one 128-byte run of global memory, B narrower for long lines):
//   k_fft_mr_lines    strided complex lines (y and x passes), in place or out of place, forward or inverse
//   k_fft_mr_z_r2c    real rows of even Nz -> packed complex FFT of M = Nz/2 (M may be odd) -> Hermitian split, Nz/2+1 modes
//   k_fft_mr_z_c2r    the inverse: Hermitian merge -> packed FFT -> real rows
// The transform is an in-place decimation-in-frequency sequence of radix-8 / 4 / 2 stages for the power-of-two part and
// radix-7 / 5 / 3 stages (compile-time constants) for the rest, butterflies in registers; the store reads frequency k
// from its mixed-radix digit-reversed position.  Twiddles come from fft.cu's f8-accurate sincospi table (get_twiddle),
// staged in shared memory when it fits beside the tile.
#include "fft_common.cuh"

#define NBK_MR_MAX_STAGES 16
#define NBK_MR_MAX_LINE 8192

// factor plan of a line of length N: stage s transforms blocks of span[s] elements with radix r[s] (q[s] = span[s] / r[s]
// butterflies per block); its twiddles are tw[m * q * tws[s]] of a table of twmul * N entries
struct MrPlan {
    int ns;
    int r[NBK_MR_MAX_STAGES], span[NBK_MR_MAX_STAGES], q[NBK_MR_MAX_STAGES], tws[NBK_MR_MAX_STAGES];
};

static bool is_smooth7(int64_t n) {
    if (n < 1) return false;
    for (int p : {2, 3, 5, 7})
        while (n % p == 0) n /= p;
    return n == 1;
}

// twmul: the table has twmul * N entries (1 for the line passes, 2 for the z passes, which share the W_Nz table)
static MrPlan make_plan(int N, int twmul) {
    MrPlan p;
    p.ns = 0;
    int rem = N, span = N, e2 = 0;
    auto push = [&](int r) {
        p.r[p.ns] = r; p.span[p.ns] = span; p.q[p.ns] = span / r; p.tws[p.ns] = twmul * (N / span);
        span /= r;
        p.ns++;
    };
    while (rem % 2 == 0) { rem /= 2; e2++; }
    for (; e2 >= 3; e2 -= 3) push(8);
    if (e2 == 2) push(4);
    else if (e2 == 1) push(2);
    for (int f : {7, 5, 3})
        while (rem % f == 0) { rem /= f; push(f); }
    return p;
}

// ---- butterflies ---------------------------------------------------------------------------------------------------
// cos / sin (2 pi i / R) for the odd radices; after unrolling every index is a compile-time constant
template <int R> __device__ __forceinline__ double cos_r(int i);
template <int R> __device__ __forceinline__ double sin_r(int i);
template <> __device__ __forceinline__ double cos_r<3>(int i) { return i == 0 ? 1.0 : -0.5; }
template <> __device__ __forceinline__ double sin_r<3>(int i) { return i == 0 ? 0.0 : (i == 1 ? 0.86602540378443864676 : -0.86602540378443864676); }
template <> __device__ __forceinline__ double cos_r<5>(int i) {
    return i == 0 ? 1.0 : (i == 1 || i == 4) ? 0.30901699437494742410 : -0.80901699437494742410;
}
template <> __device__ __forceinline__ double sin_r<5>(int i) {
    return i == 0 ? 0.0 : i == 1 ? 0.95105651629515357212 : i == 2 ? 0.58778525229247312917
                        : i == 3 ? -0.58778525229247312917 : -0.95105651629515357212;
}
template <> __device__ __forceinline__ double cos_r<7>(int i) {
    return i == 0 ? 1.0 : (i == 1 || i == 6) ? 0.62348980185873353053
                        : (i == 2 || i == 5) ? -0.22252093395631440429 : -0.90096886790241912624;
}
template <> __device__ __forceinline__ double sin_r<7>(int i) {
    return i == 0 ? 0.0 : i == 1 ? 0.78183148246802980871 : i == 2 ? 0.97492791218182360702 : i == 3 ? 0.43388373911755812048
                        : i == 4 ? -0.43388373911755812048 : i == 5 ? -0.97492791218182360702 : -0.78183148246802980871;
}

// odd-R forward DFT with the conjugate-pair symmetry: for m = 1 .. (R-1)/2
//   X_m, X_{R-m} = a_0 + sum_j cos(2 pi j m / R) (a_j + a_{R-j})  -/+  i sum_j sin(2 pi j m / R) (a_j - a_{R-j})
template <int R, typename C>
__device__ __forceinline__ void dft_odd(C (&a)[R]) {
    typedef decltype(a[0].x) T;
    constexpr int H = (R - 1) / 2;
    C s[H], d[H];
    C x0 = a[0];
#pragma unroll
    for (int j = 1; j <= H; j++) {
        s[j - 1] = cadd(a[j], a[R - j]);
        d[j - 1] = csub(a[j], a[R - j]);
        x0 = cadd(x0, s[j - 1]);
    }
#pragma unroll
    for (int m = 1; m <= H; m++) {
        C A = a[0], Bs = C{0, 0};
#pragma unroll
        for (int j = 1; j <= H; j++) {
            const T c = (T)cos_r<R>((j * m) % R), sn = (T)sin_r<R>((j * m) % R);
            A.x += c * s[j - 1].x; A.y += c * s[j - 1].y;
            Bs.x += sn * d[j - 1].x; Bs.y += sn * d[j - 1].y;
        }
        a[m] = C{A.x + Bs.y, A.y - Bs.x};          // A - i Bs
        a[R - m] = C{A.x - Bs.y, A.y + Bs.x};      // A + i Bs
    }
    a[0] = x0;
}

template <int R, typename C> __device__ __forceinline__ void dft_r(C (&a)[R]) {
    if constexpr (R == 8) radix8(a);
    else if constexpr (R == 4) dft4(a[0], a[1], a[2], a[3]);
    else if constexpr (R == 2) { C x0 = a[0], x1 = a[1]; a[0] = cadd(x0, x1); a[1] = csub(x0, x1); }
    else dft_odd<R>(a);
}

// one radix-R DIF stage over B side-by-side lines of length N in shared memory (rows padded to PITCH elements):
// block blk, butterfly q takes elements blk*Ns + q + j*Q, j < R, and leaves X_m * W_Ns^{q m} at blk*Ns + q + m*Q
template <typename C, int R, int B, int PITCH>
__device__ __forceinline__ void mr_stage(C *sm, const C *tw, int N, int Ns, int Q, int tws) {
    const int work = (N / R) * B;
    for (int w = threadIdx.x; w < work; w += blockDim.x) {
        const int b = w % B, t = w / B;
        const int blk = t / Q, q = t - blk * Q;
        C *p = sm + (blk * Ns + q) * PITCH + b;
        C a[R];
#pragma unroll
        for (int j = 0; j < R; j++) a[j] = p[j * Q * PITCH];
        dft_r<R>(a);
        p[0] = a[0];
        const int ti = q * tws;
#pragma unroll
        for (int m = 1; m < R; m++) p[m * Q * PITCH] = ti ? cmul(a[m], tw[m * ti]) : a[m];
    }
}

template <typename C, int B, int PITCH>
__device__ __forceinline__ void mr_transform(C *sm, const C *tw, const MrPlan &plan, int N) {
    for (int s = 0; s < plan.ns; s++) {
        const int Ns = plan.span[s], Q = plan.q[s], tws = plan.tws[s];
        switch (plan.r[s]) {
            case 8: mr_stage<C, 8, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
            case 4: mr_stage<C, 4, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
            case 2: mr_stage<C, 2, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
            case 3: mr_stage<C, 3, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
            case 5: mr_stage<C, 5, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
            default: mr_stage<C, 7, B, PITCH>(sm, tw, N, Ns, Q, tws); break;
        }
        __syncthreads();
    }
}

// position of frequency k after the DIF stages: digit s of k (radix r[s], least significant first) selects the
// sub-block of stage s, pos = sum_s digit_s * q[s]
__device__ __forceinline__ int mr_pos(int k, const MrPlan &plan) {
    int pos = 0;
    for (int s = 0; s < plan.ns; s++) {
        int d;
        switch (plan.r[s]) {
            case 8: d = k & 7; k >>= 3; break;
            case 4: d = k & 3; k >>= 2; break;
            case 2: d = k & 1; k >>= 1; break;
            case 3: d = k % 3; k /= 3; break;
            case 5: d = k % 5; k /= 5; break;
            default: d = k % 7; k /= 7; break;
        }
        pos += d * plan.q[s];
    }
    return pos;
}

template <typename C>
__device__ __forceinline__ const C *mr_twiddles(C *sdst, const C *__restrict__ twg, int len, int stage) {
    if (!stage) return twg;
    for (int i = threadIdx.x; i < len; i += blockDim.x) sdst[i] = twg[i];
    __syncthreads();    // (stage is uniform across the CTA)
    return sdst;
}

// ---------------------------------------------------------------------------------------------------------------------
// strided line pass: element (outer, n, inner) = data[outer*outer_stride + n*line_stride + inner], inner < n_inner
// contiguous; a tile is B adjacent inner columns of one outer index.  dst == src is safe (a CTA reads its whole tile
// before it writes it back).
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int B>
__global__ void __launch_bounds__(512)
k_fft_mr_lines(const typename C2<T>::type *src, typename C2<T>::type *dst, const typename C2<T>::type *__restrict__ twg,
               const __grid_constant__ MrPlan plan, int N, int64_t line_stride, int64_t n_inner, int64_t tiles_inner,
               int64_t n_tiles, int64_t outer_stride, int stage_tw, int inverse, T scale) {
    typedef typename C2<T>::type C;
    constexpr int PITCH = B > 1 ? B + 1 : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const C *tw = mr_twiddles<C>(sm + (size_t)N * PITCH, twg, N, stage_tw);
    const T sgn = inverse ? (T)-1 : (T)1;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t outer = tile / tiles_inner;
        const int64_t inner0 = (tile - outer * tiles_inner) * B;
        const int bvalid = (int)((n_inner - inner0) < B ? (n_inner - inner0) : B);
        const C *ib = src + outer * outer_stride + inner0;
#pragma unroll 4
        for (int w = threadIdx.x; w < N * B; w += blockDim.x) {
            const int b = w % B, n = w / B;
            C v = C{0, 0};
            if (b < bvalid) v = ib[(int64_t)n * line_stride + b];
            sm[n * PITCH + b] = C{v.x, v.y * sgn};
        }
        __syncthreads();
        mr_transform<C, B, PITCH>(sm, tw, plan, N);
        C *ob = dst + outer * outer_stride + inner0;
        for (int w = threadIdx.x; w < N * B; w += blockDim.x) {
            const int b = w % B, k = w / B;
            if (b < bvalid) {
                const C v = sm[mr_pos(k, plan) * PITCH + b];
                ob[(int64_t)k * line_stride + b] = C{v.x * scale, v.y * sgn * scale};
            }
        }
        __syncthreads();        // the next tile overwrites the buffer
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// z pass forward: real rows [rows][Nz] -> complex rows [rows][Nz/2+1], scaled by `scale`.  A tile is B rows; the
// packed pairs z[n] = x[2n] + i x[2n+1] of row b land in column b of the tile (lanes along the row).
// ---------------------------------------------------------------------------------------------------------------------
template <typename T, int B>
__global__ void __launch_bounds__(512)
k_fft_mr_z_r2c(const T *__restrict__ real, typename C2<T>::type *__restrict__ cplx,
               const typename C2<T>::type *__restrict__ twg, const __grid_constant__ MrPlan plan, int Nz, int64_t rows,
               int stage_tw, T scale) {
    typedef typename C2<T>::type C;
    constexpr int PITCH = B > 1 ? B + 1 : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const int M = Nz >> 1, Nzc = M + 1;
    const C *tw = mr_twiddles<C>(sm + (size_t)M * PITCH, twg, Nz, stage_tw);     // W_Nz^k; W_M^j = W_Nz^2j
    const int64_t n_tiles = (rows + B - 1) / B;
    const T h = (T)0.5 * scale;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * B;
        const int bvalid = (int)((rows - row0) < B ? (rows - row0) : B);
        const C *src = reinterpret_cast<const C *>(real + row0 * Nz);
#pragma unroll 4
        for (int w = threadIdx.x; w < M * B; w += blockDim.x) {
            const int b = w / M, n = w - b * M;
            sm[n * PITCH + b] = b < bvalid ? src[(int64_t)b * M + n] : C{0, 0};
        }
        __syncthreads();
        mr_transform<C, B, PITCH>(sm, tw, plan, M);
        C *dst = cplx + row0 * Nzc;
        for (int w = threadIdx.x; w < Nzc * B; w += blockDim.x) {
            const int b = w / Nzc, k = w - b * Nzc;
            if (b < bvalid) {
                const C zk = sm[mr_pos(k == M ? 0 : k, plan) * PITCH + b];
                const C zm = cconj(sm[mr_pos(k == 0 ? 0 : M - k, plan) * PITCH + b]);
                dst[(int64_t)b * Nzc + k] = hermitian_split(zk, zm, tw[k], h);
            }
        }
        __syncthreads();
    }
}

// z pass backward: complex rows [rows][Nz/2+1] -> real rows [rows][Nz], unnormalised (times `scale`)
template <typename T, int B>
__global__ void __launch_bounds__(512)
k_fft_mr_z_c2r(const typename C2<T>::type *__restrict__ cplx, T *__restrict__ real,
               const typename C2<T>::type *__restrict__ twg, const __grid_constant__ MrPlan plan, int Nz, int64_t rows,
               int stage_tw, T scale) {
    typedef typename C2<T>::type C;
    constexpr int PITCH = B > 1 ? B + 1 : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C *sm = reinterpret_cast<C *>(smem_raw);
    const int M = Nz >> 1, Nzc = M + 1;
    const C *tw = mr_twiddles<C>(sm + (size_t)M * PITCH, twg, Nz, stage_tw);
    const int64_t n_tiles = (rows + B - 1) / B;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * B;
        const int bvalid = (int)((rows - row0) < B ? (rows - row0) : B);
        const C *src = cplx + row0 * Nzc;
        for (int w = threadIdx.x; w < M * B; w += blockDim.x) {
            const int b = w / M, k = w - b * M;
            C v = C{0, 0};
            if (b < bvalid) v = hermitian_merge(src[(int64_t)b * Nzc + k], cconj(src[(int64_t)b * Nzc + (M - k)]), tw[k]);
            sm[k * PITCH + b] = v;
        }
        __syncthreads();
        mr_transform<C, B, PITCH>(sm, tw, plan, M);
        C *dst = reinterpret_cast<C *>(real + row0 * Nz);
        for (int w = threadIdx.x; w < M * B; w += blockDim.x) {
            const int b = w / M, n = w - b * M;
            if (b < bvalid) {
                const C v = sm[mr_pos(n, plan) * PITCH + b];
                dst[(int64_t)b * M + n] = C{v.x * scale, -v.y * scale};
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// launch geometry
// ---------------------------------------------------------------------------------------------------------------------
struct MrLaunch {
    int B, nthreads, stage_tw;
    size_t smem;
    int64_t grid;
};

// B side-by-side lines of length N: 128-byte runs while the tile fits one SM, narrower only for long lines; two or more
// CTAs per SM while the tile is small enough (up to N ~ 768 f8), one 512-thread CTA beyond that
static MrLaunch mr_geometry(int N, size_t cs, int64_t n_cols, int table_len) {
    const size_t budget = 227 * 1024, reserve = 1024;
    auto tile_bytes = [&](int B) { return (size_t)N * (B > 1 ? B + 1 : 1) * cs; };
    MrLaunch L;
    L.B = (int)(128 / cs);
    while (L.B > 1 && (L.B / 2 >= n_cols || tile_bytes(L.B) + reserve > budget)) L.B >>= 1;
    const size_t tile = tile_bytes(L.B), table = (size_t)table_len * cs;
    int per_sm = (int)(budget / (tile + reserve));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    // twiddles in shared memory when they fit without costing a resident CTA
    L.stage_tw = (tile + table + reserve) * per_sm <= budget;
    L.smem = tile + (L.stage_tw ? table : 0);
    L.nthreads = per_sm >= 2 ? 256 : 512;
    while (L.nthreads > 64 && L.nthreads / 2 >= (int64_t)N * L.B) L.nthreads >>= 1;
    L.grid = (int64_t)NBK_SM_COUNT * per_sm;
    return L;
}

template <typename K>
static int mr_finish_grid(K kernel, MrLaunch &L, int64_t n_tiles) {
    NBK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
    int occ = 1;        // persistent tile loop: one wave of resident CTAs (registers may allow fewer than shared memory)
    NBK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, L.nthreads, L.smem));
    if (occ < 1) occ = 1;
    if (L.grid > (int64_t)NBK_SM_COUNT * occ) L.grid = (int64_t)NBK_SM_COUNT * occ;
    if (L.grid > n_tiles) L.grid = n_tiles;
    if (L.grid < 1) L.grid = 1;
    return NBK_OK;
}

template <typename T>
static int launch_mr_lines(const void *src, void *dst, int N, int64_t line_stride, int64_t n_inner, int64_t n_outer,
                           int64_t outer_stride, int inverse, double scale, cudaStream_t s) {
    typedef typename C2<T>::type C;
    void *tw;
    int rc = get_twiddle(N, sizeof(T) == 4 ? NBK_F4 : NBK_F8, s, &tw);
    if (rc) return rc;
    const MrPlan plan = make_plan(N, 1);
    MrLaunch L = mr_geometry(N, sizeof(C), n_inner, N);
    const int64_t tiles_inner = (n_inner + L.B - 1) / L.B, n_tiles = tiles_inner * n_outer;
#define LAUNCH_MRL(BB)                                                                                                 \
    case BB:                                                                                                           \
        rc = mr_finish_grid(k_fft_mr_lines<T, BB>, L, n_tiles);                                                        \
        if (rc) return rc;                                                                                             \
        k_fft_mr_lines<T, BB><<<(int)L.grid, L.nthreads, L.smem, s>>>((const C *)src, (C *)dst, (const C *)tw, plan, N,   \
            line_stride, n_inner, tiles_inner, n_tiles, outer_stride, L.stage_tw, inverse, (T)scale);                  \
        break;
    switch (L.B) {
        LAUNCH_MRL(1) LAUNCH_MRL(2) LAUNCH_MRL(4) LAUNCH_MRL(8) LAUNCH_MRL(16)
        default: nbk_set_error("fft_mr_lines: internal tile width %d", L.B); return NBK_ERR_ARG;
    }
#undef LAUNCH_MRL
    NBK_LAUNCHED();
    return NBK_OK;
}

template <typename T>
static int launch_mr_z(const void *in, void *out, int64_t rows, int Nz, bool forward, double scale, cudaStream_t s) {
    typedef typename C2<T>::type C;
    void *tw;
    int rc = get_twiddle(Nz, sizeof(T) == 4 ? NBK_F4 : NBK_F8, s, &tw);
    if (rc) return rc;
    const int M = Nz / 2;
    const MrPlan plan = make_plan(M, 2);
    MrLaunch L = mr_geometry(M, sizeof(C), rows, Nz);
    const int64_t n_tiles = (rows + L.B - 1) / L.B;
#define LAUNCH_MRZ(BB)                                                                                                 \
    case BB:                                                                                                           \
        if (forward) {                                                                                                 \
            rc = mr_finish_grid(k_fft_mr_z_r2c<T, BB>, L, n_tiles);                                                    \
            if (rc) return rc;                                                                                         \
            k_fft_mr_z_r2c<T, BB><<<(int)L.grid, L.nthreads, L.smem, s>>>((const T *)in, (C *)out, (const C *)tw, plan,   \
                                                                          Nz, rows, L.stage_tw, (T)scale);             \
        } else {                                                                                                       \
            rc = mr_finish_grid(k_fft_mr_z_c2r<T, BB>, L, n_tiles);                                                    \
            if (rc) return rc;                                                                                         \
            k_fft_mr_z_c2r<T, BB><<<(int)L.grid, L.nthreads, L.smem, s>>>((const C *)in, (T *)out, (const C *)tw, plan,   \
                                                                          Nz, rows, L.stage_tw, (T)scale);             \
        }                                                                                                              \
        break;
    switch (L.B) {
        LAUNCH_MRZ(1) LAUNCH_MRZ(2) LAUNCH_MRZ(4) LAUNCH_MRZ(8) LAUNCH_MRZ(16)
        default: nbk_set_error("fft_mr_z: internal tile width %d", L.B); return NBK_ERR_ARG;
    }
#undef LAUNCH_MRZ
    NBK_LAUNCHED();
    return NBK_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------------------
int nbk_check_mixed_dims(const char *who, int dtype, int64_t Nx, int64_t Ny, int64_t Nz) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "%s: bad dtype %d", who, dtype);
    const bool ok = Nx >= 2 && Ny >= 2 && Nz >= 2 && Nx % 2 == 0 && Ny % 2 == 0 && Nz % 2 == 0 && is_smooth7(Nx) &&
                    is_smooth7(Ny) && is_smooth7(Nz) && Nx <= 8192 && Ny <= 8192 && Nz <= 16384;
    NBK_CHECK_ARG(ok, "%s: Nmesh (%lld,%lld,%lld) unsupported: each side must be 2^a·3^b·5^c·7^d with a >= 1 "
                      "(every side even), Nx, Ny <= 8192, Nz <= 16384", who, (long long)Nx, (long long)Ny, (long long)Nz);
    return NBK_OK;
}

extern "C" int nbk_fft_mr_lines(const void *src, void *dst, int dtype, int64_t n_line, int64_t line_stride,
                                int64_t n_inner, int64_t n_outer, int64_t outer_stride, int inverse, double scale,
                                void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_mr_lines: bad dtype %d", dtype);
    NBK_CHECK_ARG(n_line >= 2 && n_line <= NBK_MR_MAX_LINE && is_smooth7(n_line),
                  "fft_mr_lines: line length %lld unsupported: must be 2^a·3^b·5^c·7^d, 2 <= n <= %d", (long long)n_line,
                  NBK_MR_MAX_LINE);
    if (n_inner <= 0 || n_outer <= 0) return NBK_OK;
    NBK_CHECK_ARG(src != nullptr && dst != nullptr, "fft_mr_lines: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4)
        return launch_mr_lines<float>(src, dst, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
    return launch_mr_lines<double>(src, dst, (int)n_line, line_stride, n_inner, n_outer, outer_stride, inverse, scale, s);
}

extern "C" int nbk_fft_mr_z(const void *src, void *dst, int dtype, int64_t rows, int64_t Nz, int inverse, double scale,
                            void *stream) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "fft_mr_z: bad dtype %d", dtype);
    NBK_CHECK_ARG(Nz >= 2 && Nz % 2 == 0 && Nz <= 2 * NBK_MR_MAX_LINE && is_smooth7(Nz),
                  "fft_mr_z: Nz %lld unsupported: must be even and 2^a·3^b·5^c·7^d, Nz <= %d", (long long)Nz,
                  2 * NBK_MR_MAX_LINE);
    if (rows <= 0) return NBK_OK;
    NBK_CHECK_ARG(src != nullptr && dst != nullptr && src != dst, "fft_mr_z: needs two distinct buffers");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == NBK_F4) return launch_mr_z<float>(src, dst, rows, (int)Nz, !inverse, scale, s);
    return launch_mr_z<double>(src, dst, rows, (int)Nz, !inverse, scale, s);
}

extern "C" int nbk_r2c_mr(const void *real, void *cplx, int dtype, const int64_t *nmesh, double extra_scale, void *stream) {
    int rc = nbk_check_mixed_dims("r2c_mr", dtype, nmesh[0], nmesh[1], nmesh[2]);
    if (rc) return rc;
    const int64_t Nx = nmesh[0], Ny = nmesh[1], Nz = nmesh[2], Nzc = Nz / 2 + 1;
    rc = nbk_fft_mr_z(real, cplx, dtype, Nx * Ny, Nz, 0, 1.0, stream);
    if (rc) return rc;
    rc = nbk_fft_mr_lines(cplx, cplx, dtype, Ny, Nzc, Nzc, Nx, Ny * Nzc, 0, 1.0, stream);
    if (rc) return rc;
    const double scale = extra_scale / ((double)Nx * (double)Ny * (double)Nz);
    return nbk_fft_mr_lines(cplx, cplx, dtype, Nx, Ny * Nzc, Ny * Nzc, 1, 0, 0, scale, stream);
}

// c2r destroys its complex input unless `work` (same size as cplx) is given; then the x pass writes into `work`
extern "C" int nbk_c2r_mr(const void *cplx, void *real, int dtype, const int64_t *nmesh, void *work, void *stream) {
    int rc = nbk_check_mixed_dims("c2r_mr", dtype, nmesh[0], nmesh[1], nmesh[2]);
    if (rc) return rc;
    const int64_t Nx = nmesh[0], Ny = nmesh[1], Nz = nmesh[2], Nzc = Nz / 2 + 1;
    void *c = (work && work != cplx) ? work : const_cast<void *>(cplx);
    rc = nbk_fft_mr_lines(cplx, c, dtype, Nx, Ny * Nzc, Ny * Nzc, 1, 0, 1, 1.0, stream);
    if (rc) return rc;
    rc = nbk_fft_mr_lines(c, c, dtype, Ny, Nzc, Nzc, Nx, Ny * Nzc, 1, 1.0, stream);
    if (rc) return rc;
    return nbk_fft_mr_z(c, real, dtype, Nx * Ny, Nz, 1, 1.0, stream);
}
