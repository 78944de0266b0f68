/*
 * nbk_b200 -- C ABI of the B200-native FFTPower hot path (libnbk_b200.so).
 *
 * The reference (bccp/nbodykit) has no C ABI of its own: its seam for this path is the
 * duck-typed Python interface of the un-vendored `pmesh` package.  Each entry point
 * below names the reference call site(s) whose arithmetic it replaces (paths relative to
 * the nbodykit tree).  All pointers are DEVICE pointers unless marked `host`; sizes are
 * element counts; every call is asynchronous and ordered on `stream` (a cudaStream_t
 * passed as void*, NULL = legacy default stream).  Return value: 0 on success, negative
 * on error (nbk_last_error() gives the text).  No torch types, no C++ exceptions cross
 * this boundary.
 */
#ifndef NBK_B200_H
#define NBK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* scalar type codes */
#define NBK_F4 4
#define NBK_F8 8

/* resampling windows: value == support (pmesh.window.methods[...].support,
 * source/mesh/catalog.py:194,271-273) */
#define NBK_WINDOW_NNB 1
#define NBK_WINDOW_CIC 2
#define NBK_WINDOW_TSC 3
#define NBK_WINDOW_PCS 4

/* compensation transfer functions (source/mesh/catalog.py:449-594) */
/* layout bits of the `transposed` argument of the Fourier-space entry points */
#define NBK_LAYOUT_TRANSPOSED 1  /* first stored axis is y: [y_n][Nx][Nzc] (what one slab transpose leaves behind) */
#define NBK_LAYOUT_FULLZ 2       /* the last axis stores all Nz modes (complex-dtype meshes, ComplexField.compressed
                                    == False, algorithms/fftpower.py:572) instead of the Hermitian half Nz/2+1 */

#define NBK_COMP_NONE 0
#define NBK_COMP_CIC 1           /* CompensateCIC            :513-535 */
#define NBK_COMP_TSC 2           /* CompensateTSC            :449-473 */
#define NBK_COMP_PCS 3           /* CompensatePCS            :475-500 */
#define NBK_COMP_CIC_SHOTNOISE 4 /* CompensateCICShotnoise   :573-594 */
#define NBK_COMP_TSC_SHOTNOISE 5 /* CompensateTSCShotnoise   :537-559 */
#define NBK_COMP_PCS_SHOTNOISE 6 /* CompensatePCSShotnoise   :561-571 */

/* error codes */
#define NBK_OK 0
#define NBK_ERR_ARG -1
#define NBK_ERR_CUDA -2
#define NBK_ERR_UNSUPPORTED -3

int nbk_version(void);
const char *nbk_last_error(void);
/* number of kernels this library has launched since load (bench.py's "gpu_launches") */
int64_t nbk_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * Layout of a (slab of a) mesh.  Real field: x-major C order [x_n][Ny][Nz].  Complex field:
 * Hermitian-compressed on the last axis, Nzc = Nz/2+1.  `transposed == 0`: [x_n][Ny][Nzc]
 * holding x planes [x_start, x_start+x_n);  `transposed == 1`: [y_n][Nx][Nzc] holding y rows
 * [y_start, y_start+y_n) of every x (what the slab FFT leaves on each GPU when P > 1).
 * ------------------------------------------------------------------------------------- */

/* pm.paint(pos, mass=, resampler=, transform=pm.affine[.shift(s)], hold=True, out=)
 * -- source/mesh/catalog.py:287,295-296 (pmesh window scatter).
 * pos: [n][3] row-major, pos_dtype F4|F8.  mass: [n] or NULL (unit), mass_dtype F4|F8.
 * Grid coordinate g_d = fl(fl(double(pos_d)*fl(N_d/L_d)) + shift) (no FMA), periodic wrap in
 * grid units; stencil points whose x plane is outside [x_start, x_start+x_n) are dropped
 * (pmesh ghost semantics).  Always accumulates into `mesh` (hold=True); zero it first
 * with nbk_fill for hold=False.  mesh_dtype F4|F8. */
int nbk_paint(const void *pos, int pos_dtype, int64_t n, const void *mass, int mass_dtype,
              int window, double shift, const double *boxsize_host, const int64_t *nmesh_host,
              int64_t x_start, int64_t x_n, void *mesh, int mesh_dtype, void *stream);

/* same, painting the un-shifted and the +0.5-cell shifted mesh in one pass over the particles
 * (the interlaced branch, source/mesh/catalog.py:289-296) */
int nbk_paint_interlaced(const void *pos, int pos_dtype, int64_t n, const void *mass,
                         int mass_dtype, int window, const double *boxsize_host,
                         const int64_t *nmesh_host, int64_t x_start, int64_t x_n, void *mesh1,
                         void *mesh2, int mesh_dtype, void *stream);

/* The same scatter through the tile-sorted path: particles are bucketed by 16^3-cell tile, each tile is
 * accumulated in shared memory in 64-bit fixed point (order-independent, resolution 2^-31 of the largest
 * |mass|) and flushed once.  mesh2 != NULL paints the +0.5-cell shifted mesh of the interlaced branch from
 * the same buckets (then shift must be 0).  `work`: device scratch of nbk_paint_tiled_workspace() bytes.
 * clear != 0 gives pm.paint(hold=False): the mesh(es) are zeroed by the call itself (inside the bucketing
 * pass, no separate fill); clear == 0 accumulates into what is there (hold=True).
 * nbk_paint_tiled_supported() says whether the mesh admits the tiling (sides multiples of 16, >= 32). */
int nbk_paint_tiled_supported(const int64_t *nmesh_host, int64_t x_n, int window);
int64_t nbk_paint_tiled_workspace(int64_t n, int pos_dtype, int mass_dtype, const int64_t *nmesh_host,
                                  int64_t x_n);
int nbk_paint_tiled(const void *pos, int pos_dtype, int64_t n, const void *mass, int mass_dtype, int window,
                    double shift, const double *boxsize_host, const int64_t *nmesh_host, int64_t x_start,
                    int64_t x_n, void *mesh, void *mesh2, int mesh_dtype, void *work, int64_t work_bytes,
                    int clear, void *stream);

/* pm.decompose(pos, smoothing) + Layout.exchange (source/mesh/catalog.py:271-284) for the x-slab decomposition:
 * nbk_route_count finds the particles with a plane within `smoothing` cells (periodic) owned by ANOTHER rank
 * (P <= 32) and appends one entry per such particle to `list` (device uint64[n] capacity, any order):
 * index in the low 32 bits, destination bitmask in the high 32 bits.  `counts`: device uint64[P+1], zero first;
 * [0..P) receive the per-destination counts, [P] the number of list entries.
 * nbk_route_scatter copies (pos[, mass]) of the listed particles into per-destination segments of a send
 * buffer (`offsets`: device int64[P] exclusive scan of the counts; `cursor`: device uint64[P], zero first);
 * `send_index` (optional, device int64[sum counts]) receives the source row of every sent row, so that per-row
 * results computed by the destination (readout partial sums) can be added back after the return all-to-all.
 * Local particles are never copied: each rank paints its own array plus what it receives. */
int nbk_route_count(const void *pos, int pos_dtype, int64_t n, double smoothing, const double *boxsize_host,
                    const int64_t *nmesh_host, int P, int rank, uint64_t *counts, uint64_t *list, void *stream);
int nbk_route_scatter(const void *pos, int pos_dtype, const void *mass, int mass_dtype, const uint64_t *list,
                      int64_t n_list, int P, const int64_t *offsets, uint64_t *cursor, void *send_pos,
                      void *send_mass, int64_t *send_index, void *stream);

/* RealField.readout(pos, resampler=, transform=, out=) (pmesh; called from algorithms/fftrecon.py:239-244): the gather
 * transposed to nbk_paint -- out[p] (= or +=, `accumulate`) sum over the stencil of W * mesh[cell], same grid
 * coordinate / window / slab semantics (planes outside [x_start, x_start+x_n) contribute nothing: per-rank partial
 * sums).  out: device [n] of out_dtype. */
int nbk_readout(const void *mesh, int mesh_dtype, const void *pos, int pos_dtype, int64_t n, int window, double shift,
                const double *boxsize_host, const int64_t *nmesh_host, int64_t x_start, int64_t x_n, void *out,
                int out_dtype, int accumulate, void *stream);

/* reconstruction displacement modes (algorithms/fftrecon.py:213-230, Field.apply(kernel(d), kind='wavenumber')):
 * out = i k_axis / k^2 * in * exp(-k^2 R^2 / 2) / (bias (1 + f/bias mu^2)), mu = k.los/|k|, the k = 0 mode -> 0.
 * Out of place on the Hermitian-compressed field (same layout flags as nbk_compensate). */
int nbk_recon_displacement(const void *in, void *out, int dtype, const int64_t *nmesh_host, const double *boxsize_host,
                           int transposed, int64_t start, int64_t count, int axis, double R, double bias, double f,
                           const double *los_host, void *stream);

/* leftmost stencil cell (wrapped) of every particle, [n][3] int32 -- the bit-exact part of the
 * paint contract, exported for parity tests and for pm.decompose (catalog.py:271-273) */
int nbk_cell_index(const void *pos, int pos_dtype, int64_t n, int window, double shift,
                   const double *boxsize_host, const int64_t *nmesh_host, int32_t *cell_out,
                   void *stream);

/* Wlocal = sum w, W2local = sum w^2 (source/mesh/catalog.py:265-267); out2: device double[2],
 * accumulated into (zero it first). */
int nbk_sum_w_w2(const void *w, int dtype, int64_t n, double *out2, void *stream);

/* RealField.r2c / ComplexField.c2r (base/mesh.py:228,237; source/mesh/catalog.py:341-351).
 * Forward is normalised by 1/(Nx*Ny*Nz), backward unnormalised (source/mesh/array.py:36-37).
 * Single-GPU whole-mesh transforms; real [Nx][Ny][Nz], cplx [Nx][Ny][Nzc].  Out of place. */
int nbk_r2c(const void *real, void *cplx, int dtype, const int64_t *nmesh_host, double extra_scale,
            void *stream); /* cplx = extra_scale * FFT(real) / prod(N): folds e.g. the 1/nbar of catalog.py:394-398 */
int nbk_c2r(const void *cplx, void *real, int dtype, const int64_t *nmesh_host, void *work,
            void *stream);

/* the three 1-D passes of the slab-decomposed transform, for the multi-GPU path (P > 1):
 *   zy pass : real slab [x_n][Ny][Nz] -> cplx slab [x_n][Ny][Nzc], r2c along z then FFT along y
 *   pack    : cplx slab [x_n][Ny][Nzc] -> send buffer [P][y_n][x_n][Nzc] (block p = y rows of rank p)
 *   x pass  : after the all-to-all the receive buffer [P][y_n][x_n][Nzc] IS [y_n][Nx][Nzc] re-ordered;
 *             unpack -> [y_n][Nx][Nzc], FFT along x, scale by `scale`.
 * and their inverses for c2r. */
int nbk_fft_zy_forward(const void *real, void *cplx, int dtype, int64_t x_n, int64_t Ny, int64_t Nz,
                       void *stream);
int nbk_fft_zy_backward(void *cplx, void *real, int dtype, int64_t x_n, int64_t Ny, int64_t Nz,
                        void *stream);
int nbk_fft_lines(void *cplx, int dtype, int64_t n_line, int64_t line_stride, int64_t n_inner,
                  int64_t n_outer, int64_t outer_stride, int inverse, double scale, void *stream);
int nbk_fft_lines_oop(const void *src, void *dst, int dtype, int64_t n_line, int64_t line_stride, int64_t n_inner,
                      int64_t n_outer, int64_t outer_stride, int inverse, double scale, void *stream);
int nbk_fft_z_forward(const void *real, void *cplx, int dtype, int64_t rows, int64_t Nz, void *stream);
/* Fused line pass + slab transpose over NVLink peer memory: FFT along the second stored axis of the local slab
 * src[n_outer][n_line][n_inner]; output frequency k is stored directly into rank (k / (n_line/P))'s buffer at
 * peer[p][((k % (n_line/P)) * (n_outer*P) + outer_start + outer) * n_inner + kz].  peer_ptrs_host: host array of P
 * device pointers valid on this GPU (CUDA IPC / symmetric memory; entry `rank` = the local buffer).  Replaces
 * y-pass write + nbk_transpose_pack + all-to-all + nbk_transpose_unpack by one kernel; the caller provides the
 * cross-rank barriers before and after. */
int nbk_fft_lines_scatter(const void *src, void *const *peer_ptrs_host, int dtype, int64_t n_line, int64_t n_inner,
                          int64_t n_outer, int64_t outer_start, int P, int inverse, double scale, void *stream);
int nbk_transpose_pack(const void *src, void *dst, int dtype, int64_t x_n, int64_t Ny, int64_t Nzc,
                       int64_t P, void *stream);
int nbk_transpose_unpack(const void *src, void *dst, int dtype, int64_t y_n, int64_t Nx,
                         int64_t Nzc, int64_t P, void *stream);
int nbk_transpose_pack_back(const void *src, void *dst, int dtype, int64_t y_n, int64_t Nx,
                            int64_t Nzc, int64_t P, void *stream);
int nbk_transpose_unpack_back(const void *src, void *dst, int dtype, int64_t x_n, int64_t Ny,
                              int64_t Nzc, int64_t P, void *stream);

/* Field.apply(func=Compensate*, kind='circular', out=Ellipsis) -- base/mesh.py:306-313 with
 * source/mesh/catalog.py:449-594.  In place on a complex slab. */
int nbk_compensate(void *cplx, int dtype, int kind, const int64_t *nmesh_host, int transposed,
                   int64_t start, int64_t count, void *stream);

/* s1 = 0.5*s1 + 0.5*s2*exp(0.5j * sum_i k_i H_i) -- source/mesh/catalog.py:345-347 */
int nbk_interlace_combine(void *c1, const void *c2, int dtype, const int64_t *nmesh_host,
                          const double *boxsize_host, int transposed, int64_t start, int64_t count,
                          void *stream);

/* FFTBase._compute_3d_power (algorithms/fftpower.py:115-128: c1*conj(c2), zero mode, *V) fused
 * with project_to_basis (:507-701) and MeshSlab.norm2/mu/hermitian_weights (meshtools.py:104-215).
 * c2 == NULL -> auto power.  If is_p3d != 0 the input is taken as an already-formed 3-D statistic
 * y3d (project_to_basis semantics only; c2, volume, clear_zero ignored).
 * k2edges: host double[Nx+1] = kedges**2; muedges: host double[Nmu+1]; ells: host int[Nell]
 * (ells[0] must be 0).  coord_dtype NBK_F4 (fixture-faithful) | NBK_F8.
 * comp1 / comp2 (NBK_COMP_*): window compensation applied on the fly to c1 / c2 (the fused equivalent of
 * running nbk_compensate on each field first); NBK_COMP_NONE when the fields are already compensated.
 * hermitian: 0 full field, 1 Hermitian-compressed last axis with y(-k) = conj y(k), 2 compressed with
 * y(-k) = -conj y(k) (the odd multipoles of ConvolvedFFTPower, A0 conj(A_l): what the reference obtains from a full
 * 'c16' mesh, convpower/catalog.py:169-176); the mirror half is folded in accordingly.
 * real_input != 0: c1 is a REAL [count][D1][Nz] statistic (FFTCorr, algorithms/fftcorr.py:148-176; needs is_p3d,
 * hermitian == 0).  coord_unit_host: per-axis coordinate of index 1 (NULL -> 2 pi / L, the wavenumbers; FFTCorr
 * passes the cell size L/N so that coordinates are the wrapped separations).
 * Outputs (device, ACCUMULATED into; zero first), nb = (Nx+2)*(Nmu+2):
 *   nsum int64[nb]; xsum, musum double[nb]; ysum double[Nell][nb][2] (re, im).  * musum may be NULL when the caller never reads the per-bin sum of mu (FFTPower mode='1d'): that reduction is then skipped. */
int nbk_power_bin(const void *c1, const void *c2, int dtype, int is_p3d, double volume,
                  int clear_zero, const int64_t *nmesh_host, const double *boxsize_host,
                  int transposed, int64_t start, int64_t count, int coord_dtype,
                  const double *k2edges_host, int Nx, const double *muedges_host, int Nmu,
                  const double *los_host, const int *ells_host, int Nell, int hermitian, int comp1,
                  int comp2, int real_input, const double *coord_unit_host, int64_t *nsum, double *xsum, double *musum, double *ysum, void *stream);

/* nbk_power_bin with a third field: c2_mirror stands for c2 at the UNSTORED mirror mode -k of every mode with
 * 0 < j_z < N_z/2, i.e. the mirror's share of the sum is conj(c1 conj(c2_mirror)) V instead of the (anti-)Hermitian
 * fold of c1 conj(c2).  This is what a full complex ('c16') mesh gives the reference when c2 carries a factor that is
 * not parity-symmetric on the Nyquist planes -- A_l = sum_m Y_lm(khat) FFT[F Y_lm] of ConvolvedFFTPower
 * (algorithms/convpower/fkp.py:571-623; convpower/catalog.py:169-176): the mirror of index N/2 keeps the label -N/2
 * (meshtools.py:150-153), so Y_lm(khat) at the mirror is not (-1)^l Y_lm(khat).  hermitian must be 1. */
int nbk_power_bin2(const void *c1, const void *c2, const void *c2_mirror, int dtype, int is_p3d, double volume,
                   int clear_zero, const int64_t *nmesh_host, const double *boxsize_host,
                   int transposed, int64_t start, int64_t count, int coord_dtype,
                   const double *k2edges_host, int Nx, const double *muedges_host, int Nmu,
                   const double *los_host, const int *ells_host, int Nell, int hermitian, int comp1,
                   int comp2, int real_input, const double *coord_unit_host, int64_t *nsum, double *xsum, double *musum, double *ysum, void *stream);

/* out = c1 * conj(c2) * scale with element 0 cleared when clear_first != 0 (the k = 0 mode on the rank that owns
 * it): FFTBase._compute_3d_power (algorithms/fftpower.py:115-128), materialised only where the 3-D power itself
 * is needed (FFTCorr, algorithms/fftcorr.py:148-150).  c2 == NULL -> auto power.  out may alias c1. */
int nbk_cross_power(const void *c1, const void *c2, void *out, int dtype, int64_t n_complex, double scale,
                    int clear_first, void *stream);

/* ConvolvedFFTPower's spherical-harmonic passes (algorithms/convpower/fkp.py:571-597), real Y_lm, l <= 8:
 *   out(x) = in(x) * Y_lm(xhat), x = wrapped grid coordinate [-L/2, L/2) + offset[3] (BoxCenter + H/2, :457);
 *   acc(k) += c(k) * Y_lm(khat), khat := 0 at k = 0 (:537). */
int nbk_ylm_mul_real(const void *in, void *out, int dtype, int l, int m, const int64_t *nmesh_host,
                     const double *boxsize_host, const double *offset_host, int64_t x_start, int64_t x_n,
                     void *stream);
int nbk_ylm_mul_complex_acc(void *acc, const void *c, int dtype, int l, int m, const int64_t *nmesh_host,
                            const double *boxsize_host, int transposed, int64_t start, int64_t count,
                            void *stream);

/* nbk_ylm_mul_complex_acc plus a second accumulator evaluated with the direction the mirror mode -k carries on a full
 * complex mesh: every component flips sign except those at the Nyquist index (label stays -N/2) -- the c2_mirror of
 * nbk_power_bin2. */
int nbk_ylm_mul_complex_acc2(void *acc, void *acc_mirror, const void *c, int dtype, int l, int m,
                             const int64_t *nmesh_host, const double *boxsize_host, int transposed, int64_t start,
                             int64_t count, void *stream);

/* Complex-dtype meshes (ParticleMesh(dtype='c16'/'c8'), base/mesh.py:50; convpower/catalog.py:151-176): pmesh keeps all
 * N^3 modes of the c2c transform.  The configuration-space fields of this path are real-valued, so the full spectrum
 * is the Hermitian completion of the r2c result: full[Nx][Ny][Nz] <- comp[Nx][Ny][Nz/2+1] (single GPU), and the
 * stored half is cut back out before a c2r (rows = planes * Ny of this rank).  nbk_hermitian_expand takes power-of-two
 * sides and the even 2^a 3^b 5^c 7^d sides of the mixed-radix transforms. */
int nbk_hermitian_expand(const void *comp, void *full, int dtype, const int64_t *nmesh_host, void *stream);
int nbk_hermitian_compress(const void *full, void *comp, int dtype, int64_t rows, int64_t Nz, void *stream);

/* Slab transpose as a line pass into P contiguous local send blocks send[p][k % (N/P)][outer][inner] followed by one
 * strided bulk copy per peer (cudaMemcpy2DAsync over NVLink, rows of n_outer * n_inner elements): the alternative to
 * nbk_fft_lines_scatter's fine-grained remote stores for the pencil transpose of pfft (r2c / c2r, base/mesh.py:228,237).
 * nbk_slab_push: block p of `send` -> rank p's field [rows_per_peer][n_outer * P][n_inner] at offset outer_start. */
int nbk_fft_lines_pack(const void *src, void *send, int dtype, int64_t n_line, int64_t n_inner, int64_t n_outer, int P,
                       int inverse, double scale, void *stream);
int nbk_slab_push(const void *send, void *const *peer_ptrs_host, int dtype, int64_t rows_per_peer, int64_t n_outer,
                  int64_t n_inner, int64_t outer_start, int P, int rank, void *stream);
/* the same two steps restricted to the outer sub-range [o0, o0 + o_cnt) of the slab (planes of x in r2c, base/mesh.py:237):
 * the caller pushes one part over NVLink on a second stream while the line pass of the next part runs */
int nbk_fft_lines_pack_range(const void *src, void *send, int dtype, int64_t n_line, int64_t n_inner, int64_t n_outer,
                             int64_t o0, int64_t o_cnt, int P, int inverse, double scale, void *stream);
int nbk_slab_push_range(const void *send, void *const *peer_ptrs_host, int dtype, int64_t rows_per_peer, int64_t n_outer,
                        int64_t n_inner, int64_t outer_start, int64_t o0, int64_t o_cnt, int P, int rank, void *stream);

/* Mixed-radix transforms for mesh sides N = 2^a 3^b 5^c 7^d (meshes such as 384, 768, 1000, 1536 per side; pmesh/pfft
 * transform any size, base/mesh.py:228,237).  Same layout, normalisation and precision as nbk_r2c / nbk_c2r and the line
 * passes above; RealField.r2c / ComplexField.c2r call these only when a side is not a power of two.  They accept powers of
 * two as well.  Every entry point validates before any CUDA call; sizes: lines 2 <= n_line <= 8192, any 7-smooth length
 * (a line pass is complex-to-complex); z pass Nz even, 7-smooth, <= 16384; whole mesh every side even and 7-smooth,
 * Nx, Ny <= 8192, Nz <= 16384.
 *   nbk_fft_mr_lines : strided batched complex lines, element (outer, n, inner) at
 *                      outer*outer_stride + n*line_stride + inner (the addressing of nbk_fft_lines); src == dst is in
 *                      place; inverse != 0 is the unnormalised backward transform; the output is multiplied by scale.
 *   nbk_fft_mr_z     : inverse == 0: real rows [rows][Nz] -> complex rows [rows][Nz/2+1]; inverse != 0: the reverse
 *                      (unnormalised); times scale.  src and dst must be distinct buffers.
 *   nbk_r2c_mr / nbk_c2r_mr : the single-GPU whole-mesh transforms, parameters as nbk_r2c / nbk_c2r (nbk_c2r_mr
 *                      destroys its input unless `work`, the size of cplx, is given). */
int nbk_fft_mr_lines(const void *src, void *dst, int dtype, int64_t n_line, int64_t line_stride, int64_t n_inner,
                     int64_t n_outer, int64_t outer_stride, int inverse, double scale, void *stream);
int nbk_fft_mr_z(const void *src, void *dst, int dtype, int64_t rows, int64_t Nz, int inverse, double scale,
                 void *stream);
int nbk_r2c_mr(const void *real, void *cplx, int dtype, const int64_t *nmesh_host, double extra_scale, void *stream);
int nbk_c2r_mr(const void *cplx, void *real, int dtype, const int64_t *nmesh_host, void *work, void *stream);

/* Fourier-space resampling to another mesh size: pmesh `Field.resample`, called by MeshSource.compute(Nmesh=...)
 * (base/mesh.py:317-327).  Modes both meshes represent are copied (same integer frequency label per axis, Nyquist
 * negative), everything else in dst is zero.  Hermitian-compressed single-GPU layouts [Nx][Ny][Nz/2+1]. */
int nbk_resample_complex(const void *src, void *dst, int dtype, const int64_t *nmesh_src_host,
                         const int64_t *nmesh_dst_host, void *stream);

/* Friends-of-friends groups (FOF, algorithms/fof.py: kdcount `cluster.fof` in _fof_local :289-309, equiv_class :538-607,
 * centerofmass :647-700).  Two rows are friends when their squared separation, evaluated in f64 from the stored
 * positions, is <= ll^2; periodic calls use the minimum-image difference per axis (box_host = the three periods), a
 * NULL box means non-periodic and then lo_host / hi_host (the data bounds) place the cell grid.  Positions are [n][3]
 * rows of pos_dtype F4|F8, 0 <= n <= 2^31-1 (int32 union-find), ll > 0.  Every call checks its arguments before any
 * CUDA call.  The call sequence is workspace -> bucket -> link -> compress -> minid:
 *   nbk_fof_workspace : bytes of scratch the other calls need for this (n, ll, box | bounds); ncell_host (optional,
 *                       host int64[3]) receives the cell grid: cells of side >= ll, at most max(27, 2n) of them (the
 *                       side grows beyond ll when the cap binds).  Negative on a rejected argument.
 *   nbk_fof_bucket    : counting sort of the rows by cell.  order: int32[n], row of every sorted slot (rows of one
 *                       cell are adjacent, in no fixed order); spos: [3][n] of pos_dtype, the positions in that order
 *                       (structure of arrays).  `work` keeps the cell starts for nbk_fof_link.
 *   nbk_fof_link      : union-find over sorted slots: each slot visits the later slots of its own cell and the 13
 *                       forward neighbour cells (neighbours that wrap onto the same cell are visited once).  parent:
 *                       int32[n], written from scratch; afterwards it is a forest whose roots are the smallest slot of
 *                       each group.  Same (dtype, n, ll, box, bounds, work) as the bucket call.
 *   nbk_fof_compress  : root: int32[n] by ROW, root[order[i]] = root slot of slot i (parent is compressed in place).
 *   nbk_fof_minid     : out[row] = min over the row's group of value[row] (value NULL: row_offset + row, the global
 *                       row index -- the `minid` of _fof_local :302-307); rootmin: int64[n] scratch.  Called again with
 *                       updated values it pushes a change to the whole local group (the merge of _fof_merge :311-337).
 *   nbk_fof_reduce    : dense per-group reductions for find_features, group g = label[row] in [0, ngroups) (label
 *                       int64[n], other values skipped).  Rows are visited as order[0..n_visit) (rows >= n skipped) or,
 *                       with order NULL, 0..n.  val: [n][dim] of val_dtype (dim 1..3) or NULL (count only).  Outputs
 *                       are ACCUMULATED into (initialise them first):
 *                         op NBK_FOF_SUM : osum f64[ngroups][dim] += val, or += (val - anchor) wrapped into
 *                                          [-L/2, L/2) on every axis when box_host is given (anchor:
 *                                          int64[ngroups][dim] keys from op MIN); ocount uint64[ngroups] (optional)
 *                                          += 1 per row.
 *                         op NBK_FOF_MIN / NBK_FOF_MAX : okey int64[ngroups][dim] = min / max of the order-preserving
 *                                          key of (double)val: bits b of the double, b >= 0 ? b : b ^ (2^63 - 1).
 *                       peak / peakmax (f64[n] and int64 keys [ngroups]): a row whose peak value is below its
 *                       group's peakmax counts for group 0 instead (fof_catalog's `label1` :510). */
#define NBK_FOF_SUM 0
#define NBK_FOF_MIN 1
#define NBK_FOF_MAX 2
int64_t nbk_fof_workspace(int64_t n, double ll, const double *box_host, const double *lo_host, const double *hi_host,
                          int64_t *ncell_host);
int nbk_fof_bucket(const void *pos, int pos_dtype, int64_t n, double ll, const double *box_host, const double *lo_host,
                   const double *hi_host, void *work, int64_t work_bytes, int32_t *order, void *spos, void *stream);
int nbk_fof_link(const void *spos, int pos_dtype, int64_t n, double ll, const double *box_host, const double *lo_host,
                 const double *hi_host, const void *work, int64_t work_bytes, int32_t *parent, void *stream);
int nbk_fof_compress(int32_t *parent, int64_t n, const int32_t *order, int32_t *root, void *stream);
int nbk_fof_minid(const int32_t *root, int64_t n, const int64_t *value, int64_t row_offset, int64_t *rootmin,
                  int64_t *out, void *stream);
int nbk_fof_reduce(int op, const int64_t *label, int64_t n, const int32_t *order, int64_t n_visit, const void *val,
                   int val_dtype, int dim, const int64_t *anchor, const double *box_host, const double *peak,
                   const int64_t *peakmax, int64_t ngroups, double *osum, int64_t *okey, int64_t *ocount, void *stream);

/* Pair counts in a simulation box (SimulationBoxPairCount, algorithms/pair_counters/simbox.py; Corrfunc theory DD,
 * DDsmu, DDrppi).  Both catalogues are bucketed on ONE cell grid, planned from (n2, r_max, box_host | lo_host,
 * hi_host): cells of side >= r_max / 2, at most max(125, 2 n2) of them (the side grows when the cap binds).  A NULL box
 * means non-periodic, and then lo/hi (the joint data bounds of both catalogues) place the grid.  r_max is the largest
 * edge, or sqrt(rp_max^2 + pimax^2) in projected mode.  0 <= n <= 2^31-1.  Every call checks its arguments before any
 * CUDA call.  The call sequence is workspace -> bucket (once per catalogue, or per chunk of primaries) -> count:
 *   nbk_pc_workspace : bytes of scratch nbk_pc_bucket needs for n rows on that grid; ncell_host (optional, host
 *                      int64[3]) receives the grid.  Negative on a rejected argument.
 *   nbk_pc_stencil   : the neighbour offsets a cell visits, packed (ox+2)*25 + (oy+2)*5 + (oz+2), written to host
 *                      int32[125]: every offset of the 5x5x5 block whose cell comes closer than r_max, each cell once
 *                      when a periodic axis has fewer than 5 cells.  Returns how many (or a negative error).
 *   nbk_pc_bucket    : counting sort of one catalogue.  pos [n][3] of pos_dtype F4|F8, w [n] of w_dtype F4|F8.
 *                      spos: f64 [3][n] positions in cell order (wrapped into [0, L] when periodic), sw: f64 [n]
 *                      weights, scell: int32 [n] cell of every slot, cstart: int32 [C+1] cell starts.
 *   nbk_pc_count     : every ordered pair (primary slot, secondary slot) -> bin, ADDED to npairs uint64[nbins],
 *                      wnpairs f64[nbins] (sum of w1 w2) and sepsum f64[nbins] (sum of r, or r_p in projected mode).
 *                      Separations are float64, minimum image per axis when periodic; a pair counts when
 *                      edges[k]^2 <= d^2 < edges[k+1]^2 (edges host f64, 2 <= nedges <= 1025, edges[0] > 0, increasing).
 *                      mode NBK_PC_1D: nbins = nedges-1.  NBK_PC_2D: mu = |d_los| / d, pairs with mu >= 1 dropped,
 *                      bin (k, min(floor(mu nmu), nmu-1)), nbins = (nedges-1) nmu.  NBK_PC_PROJECTED: r_p over the two
 *                      axes other than los, pi = |d_los| < pimax (>= 1), npi = floor(pimax), bin (k, min(floor(pi npi /
 *                      pimax), npi-1)).  los in 0..2.  rmax: the r_max the buckets were planned with, at least the
 *                      largest separation a counted pair can have. */
#define NBK_PC_1D 0
#define NBK_PC_2D 1
#define NBK_PC_PROJECTED 2
int64_t nbk_pc_workspace(int64_t n, int64_t n2, double rmax, const double *box_host, const double *lo_host,
                         const double *hi_host, int64_t *ncell_host);
int nbk_pc_stencil(int64_t n2, double rmax, const double *box_host, const double *lo_host, const double *hi_host,
                   int32_t *offsets_host);
int nbk_pc_bucket(const void *pos, int pos_dtype, const void *w, int w_dtype, int64_t n, int64_t n2, double rmax,
                  const double *box_host, const double *lo_host, const double *hi_host, void *work, int64_t work_bytes,
                  double *spos, double *sw, int32_t *scell, int32_t *cstart, void *stream);
int nbk_pc_count(int mode, const double *edges_host, int nedges, int nmu, double pimax, int los, double rmax,
                 const double *spos1,
                 const double *sw1, const int32_t *scell1, const int32_t *cstart1, int64_t n1, const double *spos2,
                 const double *sw2, const int32_t *cstart2, int64_t n2, const double *box_host, const double *lo_host,
                 const double *hi_host, uint64_t *npairs, double *wnpairs, double *sepsum, void *stream);

/* elementwise helpers behind RealField/ComplexField `[...] = v`, `*= a`, `+= other`
 * (source/mesh/catalog.py:203,354,396-398; fftpower.py:128).  n counts REAL scalars. */
int nbk_fill(void *x, int dtype, int64_t n, double value, void *stream);
int nbk_scale(void *x, int dtype, int64_t n, double a, void *stream);
int nbk_axpy(void *y, const void *x, int dtype, int64_t n, double a, void *stream);
/* csum (source/mesh/catalog.py:388): out1 device double[1], accumulated into */
int nbk_sum(const void *x, int dtype, int64_t n, double *out1, void *stream);

#ifdef __cplusplus
}
#endif
#endif
