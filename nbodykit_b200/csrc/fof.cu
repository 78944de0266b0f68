// Friends-of-friends groups (nbodykit algorithms/fof.py: the kdcount `cluster.fof` of `_fof_local`, `equiv_class` and
// `centerofmass` of `fof_catalog`) for sm_100a.
//   nbk_fof_workspace : cell grid for a linking length (side >= ll on every axis, <= ~2n cells) and the scratch it needs
//   nbk_fof_bucket    : counting sort of the rows by cell -> visit order + SoA positions in that order
//   nbk_fof_link      : lock-free union-find over the own cell and the 13 forward neighbour cells (link: d^2 <= ll^2 in f64)
//   nbk_fof_compress  : path compression -> component root of every row
//   nbk_fof_minid     : component minimum of a per-row int64 value (per-root atomicMin, then a broadcast)
//   nbk_fof_reduce    : dense per-group count / sum (optionally of periodically wrapped differences) / min / max
#include "cellscan.cuh"

#define FOF_BLOCK 256

struct FofGrid {
    int nc[3];                  // cells per axis
    double lo[3];               // origin of cell 0 (0 when periodic)
    double inv[3];              // cells per unit length
    double L[3], invL[3];       // period per axis (periodic only)
    int periodic;
    double ll2;
};

static inline size_t fof_align(size_t b) { return (b + 255) & ~(size_t)255; }

// Cells per axis: floor(extent / ll), shrunk by a relative 1e-6 so that the rounding of (x - lo) * inv can never
// put two points closer than ll more than one cell apart; then coarsened until the grid has at most max(27, 2n)
// cells, so that memory stays O(n) for a small ll.
static int fof_plan(int64_t n, double ll, const double *box, const double *lo, const double *hi, FofGrid *g) {
    NBK_CHECK_ARG(n >= 0 && n <= 2147483647ll, "fof: particle count %lld out of range (0 <= n <= 2^31-1)", (long long)n);
    NBK_CHECK_ARG(ll > 0 && ll < 1e300, "fof: linking length must be > 0 and finite (got %g)", ll);
    double ext[3];
    if (box) {
        for (int d = 0; d < 3; d++)
            NBK_CHECK_ARG(box[d] > 0 && box[d] < 1e300, "fof: box sides must be > 0 (periodic) or the box NULL (non-periodic)");
        for (int d = 0; d < 3; d++) { ext[d] = box[d]; g->lo[d] = 0; g->L[d] = box[d]; g->invL[d] = 1.0 / box[d]; }
    } else {
        NBK_CHECK_ARG(lo && hi, "fof: a non-periodic call (box NULL) needs the data bounds lo and hi");
        for (int d = 0; d < 3; d++) {
            NBK_CHECK_ARG(hi[d] >= lo[d] && hi[d] - lo[d] < 1e300, "fof: bounds need lo <= hi on every axis");
            ext[d] = hi[d] - lo[d]; g->lo[d] = lo[d]; g->L[d] = 0; g->invL[d] = 0;
        }
    }
    g->periodic = box != nullptr;
    g->ll2 = ll * ll;
    // cell ids and cell starts are int32
    const double cap = n * 2.0 > 27.0 ? (n * 2.0 < 1073741824.0 ? n * 2.0 : 1073741824.0) : 27.0;
    double f = 1.0 + 1e-6;
    for (;;) {
        double tot = 1;
        for (int d = 0; d < 3; d++) {
            double c = floor(ext[d] / (ll * f));
            c = c < 1 ? 1 : (c > 1073741824.0 ? 1073741824.0 : c);
            g->nc[d] = (int)c;
            tot *= c;
        }
        if (tot <= cap) break;
        f *= 1.05;
    }
    for (int d = 0; d < 3; d++) g->inv[d] = ext[d] > 0 ? g->nc[d] / ext[d] : 0.0;
    return NBK_OK;
}

static inline int64_t fof_ncell(const FofGrid &g) { return (int64_t)g.nc[0] * g.nc[1] * g.nc[2]; }

// scratch: cell of every row int32[n] | counts / scatter cursors int32[C] | cell starts int32[C+1] | scan totals
static int64_t fof_work_bytes(int64_t n, const FofGrid &g) {
    int64_t C = fof_ncell(g), nseg = nbk_scan_nseg(C);
    return (int64_t)(fof_align(4 * (size_t)n) + fof_align(4 * (size_t)C) + fof_align(4 * (size_t)(C + 1)) +
                     fof_align(4 * (size_t)(nseg + 1)));
}

struct FofWork {
    int *cell, *cnt, *cstart, *segtot;
};

static FofWork fof_carve(void *work, int64_t n, const FofGrid &g) {
    int64_t C = fof_ncell(g);
    char *w = (char *)work;
    FofWork s;
    s.cell = (int *)w; w += fof_align(4 * (size_t)n);
    s.cnt = (int *)w; w += fof_align(4 * (size_t)C);
    s.cstart = (int *)w; w += fof_align(4 * (size_t)(C + 1));
    s.segtot = (int *)w;
    return s;
}

__device__ __forceinline__ int fof_axis_cell(double x, int d, const FofGrid &g) {
    double u;
    if (g.periodic) {
        u = x - floor(x * g.invL[d]) * g.L[d];
        u *= g.inv[d];
    } else {
        u = (x - g.lo[d]) * g.inv[d];
    }
    int c = (int)u;                       // u >= 0 up to rounding; the clamp absorbs the edges
    return c < 0 ? 0 : (c >= g.nc[d] ? g.nc[d] - 1 : c);
}

__device__ __forceinline__ int fof_cell(double x, double y, double z, const FofGrid &g) {
    return (fof_axis_cell(x, 0, g) * g.nc[1] + fof_axis_cell(y, 1, g)) * g.nc[2] + fof_axis_cell(z, 2, g);
}

template <typename T>
__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_cell(const T *__restrict__ pos, int n, FofGrid g, int *__restrict__ cell, int *__restrict__ cnt) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int c = fof_cell((double)pos[3 * (int64_t)i], (double)pos[3 * (int64_t)i + 1], (double)pos[3 * (int64_t)i + 2], g);
        cell[i] = c;
        atomicAdd(&cnt[c], 1);
    }
}

template <typename T>
__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_scatter(const T *__restrict__ pos, int n, const int *__restrict__ cell, const int *__restrict__ cstart,
              int *__restrict__ cursor, int *__restrict__ order, T *__restrict__ spos) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int c = cell[i];
        int dst = cstart[c] + atomicAdd(&cursor[c], 1);
        order[dst] = i;
        spos[dst] = pos[3 * (int64_t)i];
        spos[(int64_t)n + dst] = pos[3 * (int64_t)i + 1];
        spos[2 * (int64_t)n + dst] = pos[3 * (int64_t)i + 2];
    }
}

// ---- union-find over sorted indices; invariant parent[x] <= x, a root is its own parent ----------------------------
__device__ __forceinline__ int fof_find(int *parent, int x) {
    int cur = __ldcg(parent + x);
    if (cur != x) {
        int prev = x, next;
        while (cur > (next = __ldcg(parent + cur))) {
            parent[prev] = next;            // path halving: next is an ancestor of prev as well
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

__device__ __forceinline__ void fof_union(int *parent, int a, int b) {
    a = fof_find(parent, a);
    b = fof_find(parent, b);
    while (a != b) {
        // hook the larger root under the smaller; a failed CAS returns the new parent of the one we tried to hook
        if (a < b) {
            int r = atomicCAS(parent + b, b, a);
            if (r == b) return;
            b = fof_find(parent, r);
        } else {
            int r = atomicCAS(parent + a, a, b);
            if (r == a) return;
            a = fof_find(parent, r);
        }
    }
}

__device__ __forceinline__ double fof_diff(double a, double b, int d, const FofGrid &g) {
    double x = a - b;
    if (g.periodic) x -= g.L[d] * rint(x * g.invL[d]);      // minimum image
    return x;
}

// neighbour cell k (0..12) of the forward half of the 26-stencil, offsets 14..26 of the 27-stencil; -1 outside a
// non-periodic grid
__device__ __forceinline__ int fof_neighbour(int k, int cx, int cy, int cz, const FofGrid &g) {
    const int o = k + 14;
    int nx = cx + o / 9 - 1, ny = cy + (o / 3) % 3 - 1, nz = cz + o % 3 - 1;
    if (g.periodic) {
        nx = nx < 0 ? nx + g.nc[0] : (nx >= g.nc[0] ? nx - g.nc[0] : nx);
        ny = ny < 0 ? ny + g.nc[1] : (ny >= g.nc[1] ? ny - g.nc[1] : ny);
        nz = nz < 0 ? nz + g.nc[2] : (nz >= g.nc[2] ? nz - g.nc[2] : nz);
    } else if (nx < 0 || nx >= g.nc[0] || ny < 0 || ny >= g.nc[1] || nz < 0 || nz >= g.nc[2]) {
        return -1;
    }
    return (nx * g.nc[1] + ny) * g.nc[2] + nz;
}

template <typename T>
__global__ void __launch_bounds__(FOF_BLOCK, 4)
k_fof_link(const T *__restrict__ spos, int n, FofGrid g, const int *__restrict__ cstart, int *parent) {
    const T *xs = spos, *ys = spos + n, *zs = spos + 2 * (int64_t)n;
    // with fewer than 3 cells on a periodic axis, distinct offsets wrap onto the same cell: visit each cell once
    const bool wraps = g.periodic && (g.nc[0] < 3 || g.nc[1] < 3 || g.nc[2] < 3);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double xi = xs[i], yi = ys[i], zi = zs[i];
        const int cx = fof_axis_cell(xi, 0, g), cy = fof_axis_cell(yi, 1, g), cz = fof_axis_cell(zi, 2, g);
        const int c = (cx * g.nc[1] + cy) * g.nc[2] + cz;
        // k = -1: the later slots of the own cell; k = 0..12: the forward neighbour cells
        for (int k = -1; k < 13; k++) {
            int nb = c, jbeg = i + 1;
            if (k >= 0) {
                nb = fof_neighbour(k, cx, cy, cz, g);
                if (nb < 0 || nb == c) continue;
                if (wraps) {
                    bool dup = false;
                    for (int q = 0; q < k; q++) dup |= fof_neighbour(q, cx, cy, cz, g) == nb;
                    if (dup) continue;
                }
                jbeg = cstart[nb];
            }
            const int jend = cstart[nb + 1];
            for (int j = jbeg; j < jend; j++) {
                double dx = fof_diff((double)xs[j], xi, 0, g);
                double dy = fof_diff((double)ys[j], yi, 1, g);
                double dz = fof_diff((double)zs[j], zi, 2, g);
                if (dx * dx + dy * dy + dz * dz <= g.ll2) fof_union(parent, i, j);
            }
        }
    }
}

__global__ void __launch_bounds__(FOF_BLOCK) k_fof_iota(int *__restrict__ parent, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) parent[i] = i;
}

__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_compress(int *parent, int n, const int *__restrict__ order, int *__restrict__ root) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int r = fof_find(parent, i);
        parent[i] = r;
        root[order[i]] = r;
    }
}

__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_min_scatter(const int *__restrict__ root, int n, const long long *__restrict__ value, long long row_offset,
                  long long *__restrict__ rootmin) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        atomicMin(rootmin + root[i], value ? value[i] : row_offset + i);
}

__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_min_gather(const int *__restrict__ root, int n, const long long *__restrict__ rootmin, long long *__restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = rootmin[root[i]];
}

__global__ void __launch_bounds__(FOF_BLOCK) k_fof_fill_i64(long long *__restrict__ x, int n, long long v) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) x[i] = v;
}

// ---- dense per-group reductions ----------------------------------------------------------------------------------
// order-preserving int64 key of a double (signed compare of keys == compare of values)
__device__ __forceinline__ long long fof_key(double x) {
    long long b = __double_as_longlong(x);
    return b >= 0 ? b : b ^ 0x7fffffffffffffffll;
}
__device__ __forceinline__ double fof_unkey(long long k) {
    return __longlong_as_double(k >= 0 ? k : k ^ 0x7fffffffffffffffll);
}

struct FofReduce {
    int op, dim;
    double L[3];                 // > 0: wrap (v - anchor) into [-L/2, L/2) on that axis
    int64_t ngroups;
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_ext(long long v, bool mx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = mx ? (w > v ? w : v) : (w < v ? w : v);
    }
    return v;
}

// Rows are visited in cell order (`order`, from nbk_fof_bucket) so that a warp mostly covers one group; a warp whose 32
// rows share a group reduces in registers and issues one atomic per output, otherwise every lane issues its own.
template <typename T>
__global__ void __launch_bounds__(FOF_BLOCK)
k_fof_reduce(const long long *__restrict__ label, int64_t n, const int *__restrict__ order, int64_t n_visit,
             const T *__restrict__ val, const long long *__restrict__ anchor, const double *__restrict__ peak,
             const long long *__restrict__ peakmax, FofReduce r, double *__restrict__ osum, long long *__restrict__ okey,
             unsigned long long *__restrict__ ocnt) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t nround = ((n_visit + stride - 1) / stride) * stride;
    const int lane = threadIdx.x & 31;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nround; t += stride) {
        long long g = -1;
        int64_t row = -1;
        if (t < n_visit) {
            row = order ? (int64_t)order[t] : t;
            if (row < n) {
                g = label[row];
                if (g < 0 || g >= r.ngroups) g = -1;
                else if (peak && !(peak[row] >= fof_unkey(peakmax[g]))) g = 0;     // non-peak rows join group 0
            }
        }
        double v[3] = {0, 0, 0};
        if (g >= 0 && val) {
#pragma unroll
            for (int d = 0; d < 3; d++) {
                if (d >= r.dim) continue;
                double x = (double)val[row * r.dim + d];
                if (anchor) {
                    x -= fof_unkey(anchor[g * r.dim + d]);
                    if (r.L[d] > 0) {
                        if (x < -0.5 * r.L[d]) x += r.L[d];
                        else if (x >= 0.5 * r.L[d]) x -= r.L[d];
                    }
                }
                v[d] = x;
            }
        }
        const unsigned peers = __match_any_sync(0xffffffffu, g);
        const bool whole = peers == 0xffffffffu;
        if (whole && g < 0) continue;
        if (whole) {
            if (r.op == 0) {
#pragma unroll
                for (int d = 0; d < 3; d++) v[d] = warp_sum_d(v[d]);
            } else {
#pragma unroll
                for (int d = 0; d < 3; d++) v[d] = fof_unkey(warp_ext(fof_key(v[d]), r.op == 2));
            }
            if (lane != 0) continue;
        } else if (g < 0) {
            continue;
        }
        const unsigned long long c = whole ? 32ull : 1ull;
        if (ocnt) atomicAdd(ocnt + g, c);
#pragma unroll
        for (int d = 0; d < 3; d++) {
            if (d >= r.dim) continue;
            if (r.op == 0) atomicAdd(osum + g * r.dim + d, v[d]);
            else if (r.op == 1) atomicMin(okey + g * r.dim + d, fof_key(v[d]));
            else atomicMax(okey + g * r.dim + d, fof_key(v[d]));
        }
    }
}

// ---- C ABI -------------------------------------------------------------------------------------------------------
extern "C" int64_t nbk_fof_workspace(int64_t n, double ll, const double *box, const double *lo, const double *hi,
                                     int64_t *ncell) {
    FofGrid g;
    int rc = fof_plan(n, ll, box, lo, hi, &g);
    if (rc != NBK_OK) return rc;
    if (ncell) for (int d = 0; d < 3; d++) ncell[d] = g.nc[d];
    return fof_work_bytes(n, g);
}

static int fof_common(int dtype, int64_t n, double ll, const double *box, const double *lo, const double *hi,
                      int64_t work_bytes, FofGrid *g, const char *who) {
    NBK_CHECK_ARG(dtype == NBK_F4 || dtype == NBK_F8, "%s: position dtype %d not accepted (4 = f4 or 8 = f8)", who, dtype);
    int rc = fof_plan(n, ll, box, lo, hi, g);
    if (rc != NBK_OK) return rc;
    int64_t need = fof_work_bytes(n, *g);
    NBK_CHECK_ARG(work_bytes >= need, "%s: workspace of %lld bytes is too small (nbk_fof_workspace gives %lld)", who,
                  (long long)work_bytes, (long long)need);
    return NBK_OK;
}

extern "C" int nbk_fof_bucket(const void *pos, int dtype, int64_t n, double ll, const double *box, const double *lo,
                              const double *hi, void *work, int64_t work_bytes, int32_t *order, void *spos, void *stream) {
    FofGrid g;
    int rc = fof_common(dtype, n, ll, box, lo, hi, work_bytes, &g, "nbk_fof_bucket");
    if (rc != NBK_OK) return rc;
    if (n == 0) return NBK_OK;
    NBK_CHECK_ARG(pos && work && order && spos, "nbk_fof_bucket: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t C = fof_ncell(g);
    FofWork w = fof_carve(work, n, g);
    const int ni = (int)n, grid = nbk_grid_for(n, FOF_BLOCK, 8);
    NBK_CUDA(cudaMemsetAsync(w.cnt, 0, 4 * (size_t)C, s));
    if (dtype == NBK_F4) k_fof_cell<float><<<grid, FOF_BLOCK, 0, s>>>((const float *)pos, ni, g, w.cell, w.cnt);
    else k_fof_cell<double><<<grid, FOF_BLOCK, 0, s>>>((const double *)pos, ni, g, w.cell, w.cnt);
    NBK_LAUNCHED();
    rc = nbk_cell_scan(w.cnt, C, w.segtot, w.cstart, ni, s);
    if (rc != NBK_OK) return rc;
    NBK_CUDA(cudaMemsetAsync(w.cnt, 0, 4 * (size_t)C, s));
    if (dtype == NBK_F4) k_fof_scatter<float><<<grid, FOF_BLOCK, 0, s>>>((const float *)pos, ni, w.cell, w.cstart, w.cnt, order, (float *)spos);
    else k_fof_scatter<double><<<grid, FOF_BLOCK, 0, s>>>((const double *)pos, ni, w.cell, w.cstart, w.cnt, order, (double *)spos);
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fof_link(const void *spos, int dtype, int64_t n, double ll, const double *box, const double *lo,
                            const double *hi, const void *work, int64_t work_bytes, int32_t *parent, void *stream) {
    FofGrid g;
    int rc = fof_common(dtype, n, ll, box, lo, hi, work_bytes, &g, "nbk_fof_link");
    if (rc != NBK_OK) return rc;
    if (n == 0) return NBK_OK;
    NBK_CHECK_ARG(spos && work && parent, "nbk_fof_link: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    FofWork w = fof_carve((void *)work, n, g);
    const int ni = (int)n, grid = nbk_grid_for(n, FOF_BLOCK, 8);
    k_fof_iota<<<grid, FOF_BLOCK, 0, s>>>(parent, ni);
    NBK_LAUNCHED();
    if (dtype == NBK_F4) k_fof_link<float><<<grid, FOF_BLOCK, 0, s>>>((const float *)spos, ni, g, w.cstart, parent);
    else k_fof_link<double><<<grid, FOF_BLOCK, 0, s>>>((const double *)spos, ni, g, w.cstart, parent);
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fof_compress(int32_t *parent, int64_t n, const int32_t *order, int32_t *root, void *stream) {
    NBK_CHECK_ARG(n >= 0 && n <= 2147483647ll, "nbk_fof_compress: particle count %lld out of range (0 <= n <= 2^31-1)", (long long)n);
    if (n == 0) return NBK_OK;
    NBK_CHECK_ARG(parent && order && root, "nbk_fof_compress: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    k_fof_compress<<<nbk_grid_for(n, FOF_BLOCK, 8), FOF_BLOCK, 0, s>>>(parent, (int)n, order, root);
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fof_minid(const int32_t *root, int64_t n, const int64_t *value, int64_t row_offset, int64_t *rootmin,
                             int64_t *out, void *stream) {
    NBK_CHECK_ARG(n >= 0 && n <= 2147483647ll, "nbk_fof_minid: particle count %lld out of range (0 <= n <= 2^31-1)", (long long)n);
    NBK_CHECK_ARG(row_offset >= 0, "nbk_fof_minid: row offset must be >= 0");
    if (n == 0) return NBK_OK;
    NBK_CHECK_ARG(root && rootmin && out, "nbk_fof_minid: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const int ni = (int)n, grid = nbk_grid_for(n, FOF_BLOCK, 8);
    k_fof_fill_i64<<<grid, FOF_BLOCK, 0, s>>>((long long *)rootmin, ni, 0x7fffffffffffffffll);
    NBK_LAUNCHED();
    k_fof_min_scatter<<<grid, FOF_BLOCK, 0, s>>>(root, ni, (const long long *)value, row_offset, (long long *)rootmin);
    NBK_LAUNCHED();
    k_fof_min_gather<<<grid, FOF_BLOCK, 0, s>>>(root, ni, (const long long *)rootmin, (long long *)out);
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_fof_reduce(int op, const int64_t *label, int64_t n, const int32_t *order, int64_t n_visit,
                              const void *val, int val_dtype, int dim, const int64_t *anchor, const double *box,
                              const double *peak, const int64_t *peakmax, int64_t ngroups, double *osum, int64_t *okey,
                              int64_t *ocount, void *stream) {
    NBK_CHECK_ARG(op >= NBK_FOF_SUM && op <= NBK_FOF_MAX, "nbk_fof_reduce: op %d not accepted (0 = sum, 1 = min, 2 = max)", op);
    NBK_CHECK_ARG(n >= 0 && n_visit >= 0 && n_visit <= 2147483647ll,
                  "nbk_fof_reduce: row counts out of range (0 <= n, 0 <= n_visit <= 2^31-1)");
    NBK_CHECK_ARG(order != nullptr || n_visit == n, "nbk_fof_reduce: without a visit order n_visit must equal n");
    NBK_CHECK_ARG(ngroups >= 1, "nbk_fof_reduce: ngroups must be >= 1");
    NBK_CHECK_ARG(val == nullptr || val_dtype == NBK_F4 || val_dtype == NBK_F8,
                  "nbk_fof_reduce: value dtype %d not accepted (4 = f4 or 8 = f8)", val_dtype);
    NBK_CHECK_ARG(val == nullptr || (dim >= 1 && dim <= 3), "nbk_fof_reduce: dim %d not accepted (1, 2 or 3)", dim);
    NBK_CHECK_ARG(val != nullptr || (op == NBK_FOF_SUM && ocount != nullptr), "nbk_fof_reduce: no values: only a count (op 0 with ocount) is accepted");
    NBK_CHECK_ARG(op == NBK_FOF_SUM ? (val == nullptr || osum != nullptr) : okey != nullptr,
                  "nbk_fof_reduce: op %d needs its output (%s)", op, op == NBK_FOF_SUM ? "osum" : "okey");
    NBK_CHECK_ARG(box == nullptr || anchor != nullptr, "nbk_fof_reduce: periodic wrapping (box) needs the anchors");
    NBK_CHECK_ARG(anchor == nullptr || op == NBK_FOF_SUM, "nbk_fof_reduce: anchors apply to op 0 (sum) only");
    NBK_CHECK_ARG((peak == nullptr) == (peakmax == nullptr), "nbk_fof_reduce: peak and peakmax go together");
    FofReduce r;
    r.op = op;
    r.dim = val ? dim : 0;
    r.ngroups = ngroups;
    for (int d = 0; d < 3; d++) {
        r.L[d] = 0;
        if (box && d < dim) {
            NBK_CHECK_ARG(box[d] > 0, "nbk_fof_reduce: box sides must be > 0 (or the box NULL)");
            r.L[d] = box[d];
        }
    }
    if (n_visit == 0) return NBK_OK;
    NBK_CHECK_ARG(label != nullptr, "nbk_fof_reduce: null buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = nbk_grid_for(n_visit, FOF_BLOCK, 8);
#define FR(T) k_fof_reduce<T><<<grid, FOF_BLOCK, 0, s>>>((const long long *)label, n, order, n_visit, (const T *)val, \
        (const long long *)anchor, peak, (const long long *)peakmax, r, osum, (long long *)okey, (unsigned long long *)ocount)
    if (val_dtype == NBK_F4 && val) FR(float); else FR(double);
#undef FR
    NBK_LAUNCHED();
    return NBK_OK;
}
