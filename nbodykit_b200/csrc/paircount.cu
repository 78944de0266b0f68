// Pair counts in a simulation box (the Corrfunc theory DD / DDsmu / DDrppi calls of nbodykit
// algorithms/pair_counters/simbox.py) for sm_100a.
//   nbk_pc_workspace : cell grid for (n2, r_max, box | bounds) and the scratch nbk_pc_bucket needs for n rows
//   nbk_pc_stencil   : the neighbour offsets (in cells) whose closest distance to a cell is below r_max
//   nbk_pc_bucket    : counting sort of one catalogue by cell -> f64 SoA positions (wrapped into the box when
//                      periodic), f64 weights, the cell of every sorted slot and the cell starts
//   nbk_pc_count     : every (primary, secondary) pair of two bucketed catalogues -> histograms of pair counts,
//                      sum of w1 * w2 and sum of the first-dimension separation, ADDED to the outputs
// Both catalogues use one grid: its cell count depends on n2 and r_max, never on n1, so the primaries can be bucketed
// in chunks.  This unit is compiled with --fmad=false: the separations must be the same float64 numbers the CPU
// oracle computes, bin for bin.
#include "cellscan.cuh"

#define PC_BLOCK 128            // threads of the count kernel = primaries per work item
#define PC_TILE 128             // secondaries staged per shared-memory tile
#define PC_MAX_EDGES 1025       // squared separation edges travel as a kernel parameter
#define PC_MAX_STENCIL 125      // the 5 x 5 x 5 block
#define PC_SHARED_HIST_BYTES (40 * 1024)   // histograms up to this size live in shared memory, larger ones in global

struct PcGrid {
    int nc[3];                  // cells per axis
    double lo[3];               // origin of cell 0 (0 when periodic)
    double inv[3];              // cells per unit length
    double L[3], invL[3];       // period per axis (periodic only)
    int periodic;
};

struct PcParams {
    PcGrid g;
    int nr, nsub, nbins, los, nst;
    double pimax, inv_dpi;      // projected: pi bin = floor(pi * inv_dpi), inv_dpi = npi / pimax
    double e2[PC_MAX_EDGES];    // squared separation edges, e2[0] > 0
    int st[PC_MAX_STENCIL];     // stencil offsets, packed (ox + 2) * 25 + (oy + 2) * 5 + (oz + 2)
};

static inline size_t pc_align(size_t b) { return (b + 255) & ~(size_t)255; }

// Cells per axis: floor(extent / (r_max / 2)), shrunk by a relative 1e-6 so that rounding can never put two points
// closer than r_max more than two cells apart; then coarsened until the grid has at most max(125, 2 n2) cells.
static int pc_plan(int64_t n2, double rmax, const double *box, const double *lo, const double *hi, PcGrid *g,
                   const char *who) {
    NBK_CHECK_ARG(n2 >= 0 && n2 <= 2147483647ll, "%s: secondary count %lld out of range (0 <= n2 <= 2^31-1)", who, (long long)n2);
    NBK_CHECK_ARG(rmax > 0 && rmax < 1e300, "%s: largest separation must be > 0 and finite (got %g)", who, rmax);
    double ext[3];
    if (box) {
        for (int d = 0; d < 3; d++)
            NBK_CHECK_ARG(box[d] > 0 && box[d] < 1e300, "%s: box sides must be > 0 (periodic) or the box NULL (non-periodic)", who);
        for (int d = 0; d < 3; d++) { ext[d] = box[d]; g->lo[d] = 0; g->L[d] = box[d]; g->invL[d] = 1.0 / box[d]; }
    } else {
        NBK_CHECK_ARG(lo && hi, "%s: a non-periodic call (box NULL) needs the data bounds lo and hi", who);
        for (int d = 0; d < 3; d++) {
            NBK_CHECK_ARG(hi[d] >= lo[d] && hi[d] - lo[d] < 1e300, "%s: bounds need lo <= hi on every axis", who);
            ext[d] = hi[d] - lo[d]; g->lo[d] = lo[d]; g->L[d] = 0; g->invL[d] = 0;
        }
    }
    g->periodic = box != nullptr;
    // cell ids and cell starts are int32
    const double cap = n2 * 2.0 > 125.0 ? (n2 * 2.0 < 1073741824.0 ? n2 * 2.0 : 1073741824.0) : 125.0;
    const double side = 0.5 * rmax;
    double f = 1.0 + 1e-6;
    for (;;) {
        double tot = 1;
        for (int d = 0; d < 3; d++) {
            double c = floor(ext[d] / (side * f));
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

static inline int64_t pc_ncell(const PcGrid &g) { return (int64_t)g.nc[0] * g.nc[1] * g.nc[2]; }

// Offsets of the 5 x 5 x 5 block whose cells come closer than r_max to the centre cell (a relative 1e-6 of slack
// keeps borderline cells in).  On a periodic axis with fewer than 5 cells distinct offsets wrap onto the same cell:
// each cell is kept once.
static int pc_stencil(const PcGrid &g, double rmax, int *st) {
    double side[3];
    for (int d = 0; d < 3; d++) side[d] = g.inv[d] > 0 ? 1.0 / g.inv[d] : 0.0;
    int n = 0;
    int64_t key[PC_MAX_STENCIL];
    for (int ox = -2; ox <= 2; ox++)
        for (int oy = -2; oy <= 2; oy++)
            for (int oz = -2; oz <= 2; oz++) {
                const int o[3] = {ox, oy, oz};
                double gap2 = 0;
                int res[3];
                bool skip = false;
                for (int d = 0; d < 3; d++) {
                    const int a = o[d] < 0 ? -o[d] : o[d];
                    const double gap = a > 1 ? (a - 1) * side[d] : 0.0;
                    gap2 += gap * gap;
                    if (g.periodic) res[d] = ((o[d] % g.nc[d]) + g.nc[d]) % g.nc[d];
                    else if (a >= g.nc[d]) skip = true;          // never inside the grid
                    else res[d] = o[d] + 2;
                }
                if (skip || gap2 * (1.0 - 1e-6) >= rmax * rmax) continue;
                // the neighbour cell relative to the centre: a residue on a periodic axis, the offset otherwise
                const int64_t b1 = g.periodic ? g.nc[1] : 5, b2 = g.periodic ? g.nc[2] : 5;
                const int64_t k = (res[0] * b1 + res[1]) * b2 + res[2];
                bool dup = false;
                for (int q = 0; q < n; q++) dup |= key[q] == k;
                if (dup) continue;
                key[n] = k;
                st[n++] = (ox + 2) * 25 + (oy + 2) * 5 + (oz + 2);
            }
    return n;
}

// scratch of nbk_pc_bucket: cell of every row int32[n] | counts / scatter cursors int32[C] | scan totals
static int64_t pc_work_bytes(int64_t n, const PcGrid &g) {
    const int64_t C = pc_ncell(g);
    return (int64_t)(pc_align(4 * (size_t)n) + pc_align(4 * (size_t)C) + pc_align(4 * (size_t)(nbk_scan_nseg(C) + 1)));
}

// position on one axis as the count sees it: wrapped into [0, L] when periodic
__device__ __forceinline__ double pc_wrap(double x, int d, const PcGrid &g) {
    return g.periodic ? x - floor(x * g.invL[d]) * g.L[d] : x;
}

__device__ __forceinline__ int pc_axis_cell(double u, int d, const PcGrid &g) {
    int c = (int)((u - g.lo[d]) * g.inv[d]);      // u >= lo up to rounding; the clamp absorbs the edges
    return c < 0 ? 0 : (c >= g.nc[d] ? g.nc[d] - 1 : c);
}

template <typename T>
__global__ void __launch_bounds__(256)
k_pc_cell(const T *__restrict__ pos, int n, PcGrid g, int *__restrict__ cell, int *__restrict__ cnt) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int c = 0;
#pragma unroll
        for (int d = 0; d < 3; d++) c = c * g.nc[d] + pc_axis_cell(pc_wrap((double)pos[3 * (int64_t)i + d], d, g), d, g);
        cell[i] = c;
        atomicAdd(&cnt[c], 1);
    }
}

template <typename T, typename W>
__global__ void __launch_bounds__(256)
k_pc_scatter(const T *__restrict__ pos, const W *__restrict__ w, int n, PcGrid g, const int *__restrict__ cell,
             const int *__restrict__ cstart, int *__restrict__ cursor, double *__restrict__ spos, double *__restrict__ sw,
             int *__restrict__ scell) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int c = cell[i];
        const int dst = cstart[c] + atomicAdd(&cursor[c], 1);
#pragma unroll
        for (int d = 0; d < 3; d++) spos[d * (int64_t)n + dst] = pc_wrap((double)pos[3 * (int64_t)i + d], d, g);
        sw[dst] = (double)w[i];
        scell[dst] = c;
    }
}

__device__ __forceinline__ double pc_diff(double a, double b, int d, const PcGrid &g) {
    double x = a - b;
    if (g.periodic) x -= g.L[d] * rint(x * g.invL[d]);      // minimum image
    return x;
}

// bin k with e2[k] <= v < e2[k + 1], given e2[0] <= v < e2[nr]
__device__ __forceinline__ int pc_search(const double *e2, int nr, double v) {
    int lo = 0, hi = nr;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (v >= e2[mid]) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void pc_flush(unsigned *hc, double *hw, double *hs, int nbins, unsigned long long *gcnt,
                                         double *gw, double *gs) {
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) {
        if (hc[b]) {
            atomicAdd(gcnt + b, (unsigned long long)hc[b]);
            atomicAdd(gw + b, hw[b]);
            atomicAdd(gs + b, hs[b]);
            hc[b] = 0; hw[b] = 0; hs[b] = 0;
        }
    }
}

// One work item = PC_BLOCK consecutive sorted primary slots; the slots of one cell share the tiles of secondaries of
// every stencil cell, so a dense cell is spread over many items (and CTAs).  MODE 0 = 1d, 1 = 2d, 2 = projected.
// SH: u32 counts and f64 sums in shared memory, flushed to global before a u32 can overflow and at the end;
// otherwise global atomics.
template <int MODE, bool SH>
__global__ void __launch_bounds__(PC_BLOCK, 4)
k_pc_count(const double *__restrict__ p1, const double *__restrict__ w1, const int *__restrict__ scell1,
           const int *__restrict__ cstart1, int n1, const double *__restrict__ p2, const double *__restrict__ w2,
           const int *__restrict__ cstart2, int n2, const __grid_constant__ PcParams P,
           unsigned long long *__restrict__ gcnt, double *__restrict__ gw, double *__restrict__ gs) {
    extern __shared__ double smem[];
    double *tx = smem, *ty = tx + PC_TILE, *tz = ty + PC_TILE, *tw = tz + PC_TILE, *e2 = tw + PC_TILE;
    double *hw = e2 + (P.nr + 1), *hs = hw + P.nbins;
    unsigned *hc = (unsigned *)(hs + P.nbins);
    const int tid = threadIdx.x;
    for (int b = tid; b <= P.nr; b += PC_BLOCK) e2[b] = P.e2[b];
    if (SH) {
        for (int b = tid; b < P.nbins; b += PC_BLOCK) { hc[b] = 0; hw[b] = 0; hs[b] = 0; }
    }
    __syncthreads();
    const PcGrid &g = P.g;
    const double e2lo = P.e2[0], e2hi = P.e2[P.nr];
    const double *x1 = p1, *y1 = p1 + n1, *z1 = p1 + 2 * (int64_t)n1;
    const double *x2 = p2, *y2 = p2 + n2, *z2 = p2 + 2 * (int64_t)n2;
    const int nitems = (n1 + PC_BLOCK - 1) / PC_BLOCK;
    unsigned long long acc = 0;       // pairs evaluated since the last flush: bounds every u32 count
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        int s = item * PC_BLOCK;
        const int send = min(s + PC_BLOCK, n1);
        while (s < send) {
            const int c = scell1[s];
            const int e = min(send, cstart1[c + 1]);
            const int my = s + tid;
            const bool act = my < e;
            double xi = 0, yi = 0, zi = 0, wi = 0;
            if (act) { xi = x1[my]; yi = y1[my]; zi = z1[my]; wi = w1[my]; }
            const int cz = c % g.nc[2], cy = (c / g.nc[2]) % g.nc[1], cx = c / (g.nc[2] * g.nc[1]);
            for (int k = 0; k < P.nst; k++) {
                const int o = P.st[k];
                int nx = cx + o / 25 - 2, ny = cy + (o / 5) % 5 - 2, nz = cz + o % 5 - 2;
                if (g.periodic) {
                    nx = ((nx % g.nc[0]) + g.nc[0]) % g.nc[0];
                    ny = ((ny % g.nc[1]) + g.nc[1]) % g.nc[1];
                    nz = ((nz % g.nc[2]) + g.nc[2]) % g.nc[2];
                } else if (nx < 0 || nx >= g.nc[0] || ny < 0 || ny >= g.nc[1] || nz < 0 || nz >= g.nc[2]) {
                    continue;
                }
                const int nb = (nx * g.nc[1] + ny) * g.nc[2] + nz;
                const int j0 = cstart2[nb], j1 = cstart2[nb + 1];
                for (int t = j0; t < j1; t += PC_TILE) {
                    const int tn = min(PC_TILE, j1 - t);
                    if (SH) {
                        const unsigned long long inc = (unsigned long long)(e - s) * tn;
                        if (acc + inc > 0xffffffffull) {
                            __syncthreads();
                            pc_flush(hc, hw, hs, P.nbins, gcnt, gw, gs);
                            acc = 0;
                        }
                        acc += inc;
                    }
                    __syncthreads();                  // the previous tile is consumed (and any flush done)
                    if (tid < tn) { tx[tid] = x2[t + tid]; ty[tid] = y2[t + tid]; tz[tid] = z2[t + tid]; tw[tid] = w2[t + tid]; }
                    __syncthreads();
                    if (!act) continue;
                    for (int j = 0; j < tn; j++) {
                        const double dx = pc_diff(tx[j], xi, 0, g);
                        const double dy = pc_diff(ty[j], yi, 1, g);
                        const double dz = pc_diff(tz[j], zi, 2, g);
                        const double dl = P.los == 0 ? dx : (P.los == 1 ? dy : dz);
                        int bin;
                        double sep;
                        if (MODE == 2) {
                            const double a = P.los == 0 ? dy : dx, b = P.los == 2 ? dy : dz;
                            const double rp2 = a * a + b * b;
                            if (!(rp2 >= e2lo && rp2 < e2hi)) continue;
                            const double pi = fabs(dl);
                            if (!(pi < P.pimax)) continue;
                            int pb = (int)(pi * P.inv_dpi);
                            pb = pb < P.nsub ? pb : P.nsub - 1;
                            bin = pc_search(e2, P.nr, rp2) * P.nsub + pb;
                            sep = sqrt(rp2);
                        } else {
                            const double d2 = dx * dx + dy * dy + dz * dz;
                            if (!(d2 >= e2lo && d2 < e2hi)) continue;
                            bin = pc_search(e2, P.nr, d2);
                            sep = sqrt(d2);
                            if (MODE == 1) {
                                const double mu = fabs(dl) / sep;
                                if (!(mu < 1.0)) continue;
                                int mb = (int)(mu * P.nsub);
                                mb = mb < P.nsub ? mb : P.nsub - 1;
                                bin = bin * P.nsub + mb;
                            }
                        }
                        const double wij = wi * tw[j];
                        if (SH) {
                            atomicAdd(hc + bin, 1u);
                            atomicAdd(hw + bin, wij);
                            atomicAdd(hs + bin, sep);
                        } else {
                            atomicAdd(gcnt + bin, 1ull);
                            atomicAdd(gw + bin, wij);
                            atomicAdd(gs + bin, sep);
                        }
                    }
                }
            }
            s = e;
        }
    }
    if (SH) {
        __syncthreads();
        pc_flush(hc, hw, hs, P.nbins, gcnt, gw, gs);
    }
}

// ---- C ABI -------------------------------------------------------------------------------------------------------
extern "C" int64_t nbk_pc_workspace(int64_t n, int64_t n2, double rmax, const double *box, const double *lo,
                                    const double *hi, int64_t *ncell) {
    NBK_CHECK_ARG(n >= 0 && n <= 2147483647ll, "nbk_pc_workspace: row count %lld out of range (0 <= n <= 2^31-1)", (long long)n);
    PcGrid g;
    int rc = pc_plan(n2, rmax, box, lo, hi, &g, "nbk_pc_workspace");
    if (rc != NBK_OK) return rc;
    if (ncell) for (int d = 0; d < 3; d++) ncell[d] = g.nc[d];
    return pc_work_bytes(n, g);
}

extern "C" int nbk_pc_stencil(int64_t n2, double rmax, const double *box, const double *lo, const double *hi,
                              int32_t *offsets) {
    PcGrid g;
    int rc = pc_plan(n2, rmax, box, lo, hi, &g, "nbk_pc_stencil");
    if (rc != NBK_OK) return rc;
    NBK_CHECK_ARG(offsets != nullptr, "nbk_pc_stencil: offsets must hold 125 int32");
    int st[PC_MAX_STENCIL];
    const int n = pc_stencil(g, rmax, st);
    for (int k = 0; k < n; k++) offsets[k] = st[k];
    return n;
}

extern "C" int nbk_pc_bucket(const void *pos, int pos_dtype, const void *w, int w_dtype, int64_t n, int64_t n2,
                             double rmax, const double *box, const double *lo, const double *hi, void *work,
                             int64_t work_bytes, double *spos, double *sw, int32_t *scell, int32_t *cstart, void *stream) {
    NBK_CHECK_ARG(pos_dtype == NBK_F4 || pos_dtype == NBK_F8, "nbk_pc_bucket: position dtype %d not accepted (4 = f4 or 8 = f8)", pos_dtype);
    NBK_CHECK_ARG(w_dtype == NBK_F4 || w_dtype == NBK_F8, "nbk_pc_bucket: weight dtype %d not accepted (4 = f4 or 8 = f8)", w_dtype);
    NBK_CHECK_ARG(n >= 0 && n <= 2147483647ll, "nbk_pc_bucket: row count %lld out of range (0 <= n <= 2^31-1)", (long long)n);
    PcGrid g;
    int rc = pc_plan(n2, rmax, box, lo, hi, &g, "nbk_pc_bucket");
    if (rc != NBK_OK) return rc;
    const int64_t need = pc_work_bytes(n, g);
    NBK_CHECK_ARG(work_bytes >= need, "nbk_pc_bucket: workspace of %lld bytes is too small (nbk_pc_workspace gives %lld)",
                  (long long)work_bytes, (long long)need);
    NBK_CHECK_ARG(cstart != nullptr && work != nullptr, "nbk_pc_bucket: null buffer (work, cstart)");
    NBK_CHECK_ARG(n == 0 || (pos && w && spos && sw && scell), "nbk_pc_bucket: null buffer (pos, w, spos, sw, scell)");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t C = pc_ncell(g);
    char *wp = (char *)work;
    int *cell = (int *)wp; wp += pc_align(4 * (size_t)n);
    int *cnt = (int *)wp; wp += pc_align(4 * (size_t)C);
    int *segtot = (int *)wp;
    const int ni = (int)n, grid = nbk_grid_for(n, 256, 8);
    NBK_CUDA(cudaMemsetAsync(cnt, 0, 4 * (size_t)C, s));
    if (n) {
        if (pos_dtype == NBK_F4) k_pc_cell<float><<<grid, 256, 0, s>>>((const float *)pos, ni, g, cell, cnt);
        else k_pc_cell<double><<<grid, 256, 0, s>>>((const double *)pos, ni, g, cell, cnt);
        NBK_LAUNCHED();
    }
    rc = nbk_cell_scan(cnt, C, segtot, cstart, ni, s);
    if (rc != NBK_OK) return rc;
    if (n == 0) return NBK_OK;
    NBK_CUDA(cudaMemsetAsync(cnt, 0, 4 * (size_t)C, s));
#define PCS(T, W) k_pc_scatter<T, W><<<grid, 256, 0, s>>>((const T *)pos, (const W *)w, ni, g, cell, cstart, cnt, spos, sw, scell)
    if (pos_dtype == NBK_F4) { if (w_dtype == NBK_F4) PCS(float, float); else PCS(float, double); }
    else { if (w_dtype == NBK_F4) PCS(double, float); else PCS(double, double); }
#undef PCS
    NBK_LAUNCHED();
    return NBK_OK;
}

template <int MODE, bool SH>
static int pc_launch(const PcParams &P, size_t shmem, const double *spos1, const double *sw1, const int32_t *scell1,
                     const int32_t *cstart1, int n1, const double *spos2, const double *sw2, const int32_t *cstart2,
                     int n2, unsigned long long *npairs, double *wnpairs, double *sepsum, cudaStream_t s) {
    auto kern = k_pc_count<MODE, SH>;
    NBK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shmem));
    int occ = 0;
    NBK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, PC_BLOCK, shmem));
    const int64_t nitems = ((int64_t)n1 + PC_BLOCK - 1) / PC_BLOCK;
    const int64_t cap = (int64_t)NBK_SM_COUNT * (occ > 0 ? occ : 1);
    const int grid = (int)(nitems < cap ? nitems : cap);
    kern<<<grid, PC_BLOCK, shmem, s>>>(spos1, sw1, scell1, cstart1, n1, spos2, sw2, cstart2, n2, P, npairs, wnpairs, sepsum);
    NBK_LAUNCHED();
    return NBK_OK;
}

extern "C" int nbk_pc_count(int mode, const double *edges, int nedges, int nmu, double pimax, int los, double rmax,
                            const double *spos1, const double *sw1, const int32_t *scell1, const int32_t *cstart1,
                            int64_t n1, const double *spos2, const double *sw2, const int32_t *cstart2, int64_t n2,
                            const double *box, const double *lo, const double *hi, uint64_t *npairs, double *wnpairs,
                            double *sepsum, void *stream) {
    NBK_CHECK_ARG(mode == NBK_PC_1D || mode == NBK_PC_2D || mode == NBK_PC_PROJECTED,
                  "nbk_pc_count: mode %d not accepted (0 = 1d, 1 = 2d, 2 = projected)", mode);
    NBK_CHECK_ARG(edges != nullptr && nedges >= 2 && nedges <= PC_MAX_EDGES,
                  "nbk_pc_count: %d separation edges not accepted (2 ... %d)", nedges, PC_MAX_EDGES);
    NBK_CHECK_ARG(edges[0] > 0, "nbk_pc_count: the lowest edge must be > 0 (got %g)", edges[0]);
    for (int k = 1; k < nedges; k++)
        NBK_CHECK_ARG(edges[k] > edges[k - 1] && edges[k] < 1e150, "nbk_pc_count: edges must increase strictly and be finite");
    NBK_CHECK_ARG(los >= 0 && los <= 2, "nbk_pc_count: line of sight %d not accepted (0, 1 or 2)", los);
    NBK_CHECK_ARG(mode != NBK_PC_2D || (nmu >= 1 && nmu <= 1000000), "nbk_pc_count: 2d mode needs 1 <= nmu <= 10^6 (got %d)", nmu);
    NBK_CHECK_ARG(mode != NBK_PC_PROJECTED || (pimax >= 1 && pimax <= 1e6),
                  "nbk_pc_count: projected mode needs 1 <= pimax <= 10^6 (got %g)", pimax);
    NBK_CHECK_ARG(n1 >= 0 && n1 <= 2147483647ll && n2 >= 0 && n2 <= 2147483647ll,
                  "nbk_pc_count: row counts out of range (0 <= n1, n2 <= 2^31-1)");
    PcParams P;
    P.nr = nedges - 1;
    P.nsub = mode == NBK_PC_2D ? nmu : (mode == NBK_PC_PROJECTED ? (int)floor(pimax) : 1);
    NBK_CHECK_ARG((int64_t)P.nr * P.nsub <= (1 << 26), "nbk_pc_count: %lld bins is too many (at most 2^26)",
                  (long long)P.nr * P.nsub);
    P.nbins = P.nr * P.nsub;
    P.los = los;
    P.pimax = mode == NBK_PC_PROJECTED ? pimax : 0;
    P.inv_dpi = mode == NBK_PC_PROJECTED ? P.nsub / pimax : 0;
    const double emax = edges[nedges - 1];
    const double need = mode == NBK_PC_PROJECTED ? sqrt(emax * emax + pimax * pimax) : emax;
    NBK_CHECK_ARG(rmax >= need && rmax < 1e300, "nbk_pc_count: grid reach r_max %g is below the largest separation "
                  "%g (the largest edge, or sqrt(rp_max^2 + pimax^2) when projected)", rmax, need);
    int rc = pc_plan(n2, rmax, box, lo, hi, &P.g, "nbk_pc_count");
    if (rc != NBK_OK) return rc;
    for (int k = 0; k < nedges; k++) P.e2[k] = edges[k] * edges[k];
    P.nst = pc_stencil(P.g, rmax, P.st);
    NBK_CHECK_ARG(npairs && wnpairs && sepsum, "nbk_pc_count: null output (npairs, wnpairs, sepsum)");
    if (n1 == 0 || n2 == 0) return NBK_OK;
    NBK_CHECK_ARG(spos1 && sw1 && scell1 && cstart1 && spos2 && sw2 && cstart2, "nbk_pc_count: null input buffer");
    cudaStream_t s = (cudaStream_t)stream;
    const size_t hist = (size_t)P.nbins * (8 + 8 + 4);
    const bool sh = hist <= PC_SHARED_HIST_BYTES;
    const size_t shmem = (4 * PC_TILE + P.nr + 1) * sizeof(double) + (sh ? hist : 0);
#define PCL(M, S) pc_launch<M, S>(P, shmem, spos1, sw1, scell1, cstart1, (int)n1, spos2, sw2, cstart2, (int)n2, \
                                  (unsigned long long *)npairs, wnpairs, sepsum, s)
    if (mode == NBK_PC_1D) rc = sh ? PCL(0, true) : PCL(0, false);
    else if (mode == NBK_PC_2D) rc = sh ? PCL(1, true) : PCL(1, false);
    else rc = sh ? PCL(2, true) : PCL(2, false);
#undef PCL
    return rc;
}
