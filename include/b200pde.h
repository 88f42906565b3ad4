/* b200pde -- C ABI of the B200-native Navier2D spectral hot path.
 *
 * The reference (preiter93/rustpde-mpi) has no FFI: its seam is the Rust trait surface
 * `Space / Field / Solve / Integrate`.  Every entry point below names the reference
 * interface it replaces (paths relative to /root/reference); INTEGRATION.md shows the Rust
 * `extern "C"` binding a maintainer would add so that `Navier2D::update()` runs here.
 *
 * Conventions
 *   - opaque handles, plain pointers and sizes, no C++/torch types;
 *   - every function returns 0 on success, non-zero on error (shape mismatch, CUDA error,
 *     unsupported size) -- this replaces the reference's panics; b2_last_error() gives text;
 *   - all data stays resident on the GPU; `*_host` calls are the only H2D/D2H copies;
 *   - host arrays are row-major (ndarray default): real f64, or Complex<f64> as
 *     interleaved (re, im) pairs for spectral arrays of r2c spaces;
 *   - one CUDA stream per ctx; a handle must not be used from two threads at once.
 */
#ifndef B200PDE_H
#define B200PDE_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2_ctx b2_ctx;
typedef struct b2_space b2_space;
typedef struct b2_field b2_field;
typedef struct b2_array b2_array;
typedef struct b2_solver b2_solver;
typedef struct b2_navier b2_navier;

/* BaseKind enum order of src/field.rs:173-177 (funspace BaseKind) */
enum b2_base_kind {
  B2_CHEBYSHEV = 0,
  B2_CHEB_DIRICHLET = 1,
  B2_CHEB_NEUMANN = 2,
  B2_CHEB_DIRICHLET_NEUMANN = 3, /* bc="hc": three-term stencil, PdmaPlus2 solves (src/solver/pdma_plus2.rs) */
  B2_FOURIER_R2C = 4,
  B2_FOURIER_C2C = 5 /* not on the Navier2D path: axis 0 only, n <= 1024, dense-matrix transform, complex physical values */
};
enum b2_shape_kind { B2_SHAPE_PHYSICAL = 0, B2_SHAPE_SPECTRAL = 1, B2_SHAPE_ORTHO = 2 };
enum b2_status { B2_OK = 0, B2_ERR_ARG = 1, B2_ERR_CUDA = 2, B2_ERR_UNSUPPORTED = 3, B2_ERR_SHAPE = 4 };

const char* b2_last_error(void);
int b2_version(void);

/* ---- context: one per GPU / per rank.  Replaces funspace `initialize()`/`Universe`
 *      (src/mpi/mod.rs:5,12).  For nranks > 1 the ranks exchange a CUDA-IPC handle of one
 *      symmetric heap (b2_ctx_heap_handle / b2_ctx_attach_peers) so that the pencil transposes
 *      are peer stores fused into the producing kernel. ---- */
int b2_ctx_create(int device, int rank, int nranks, size_t heap_bytes, b2_ctx** out);
int b2_ctx_destroy(b2_ctx* ctx);
int b2_ctx_sync(b2_ctx* ctx);
/* device-side timing on the ctx stream (CUDA events): bench.py's timed region */
int b2_ctx_timer_start(b2_ctx* ctx);
int b2_ctx_timer_stop(b2_ctx* ctx, double* ms);
int b2_ctx_launch_count(const b2_ctx* ctx, long long* kernels_launched);
/* profiling aid: per-op cycle counters of the lane kernel; out64[code] = cycles, out64[32+code] = calls */
int b2_ctx_opprof(b2_ctx* ctx, int on, unsigned long long* out64);
/* memory-pipeline probe of the lane kernel (tools/copyprobe.py); not part of the reference surface */
int b2_debug_copy(b2_space* sp, int mode, int reps, double* ms);
/* read (and reset) the time spent in the dense Poisson GEMMs since profiling was switched on */
int b2_ctx_profile(b2_ctx* ctx, int on, double* gemm_ms);
int b2_ctx_heap_handle(b2_ctx* ctx, void* handle64 /* 64 bytes out */);
int b2_ctx_attach_peers(b2_ctx* ctx, const void* handles /* nranks x 64 bytes, rank order */);
/* cross-rank barrier hooks: the host (torch.distributed / MPI) calls these around its barrier */
int b2_ctx_nranks(const b2_ctx* ctx);
int b2_ctx_barrier(b2_ctx* ctx);   /* all-ranks barrier on the ctx stream (peer flags over NVLink) */

/* ---- Space2 (funspace Space2::new(&base0,&base1); src/bases.rs:11-19, src/field.rs:81-90) ---- */
int b2_space2_create(b2_ctx* ctx, int kind0, int n0, int kind1, int n1, b2_space** out);
int b2_space_destroy(b2_space* sp);
/* shape_physical / shape_spectral / ortho shape; spectral & ortho of r2c spaces are complex */
int b2_space_shape(const b2_space* sp, int shape_kind, int* rows, int* cols, int* is_complex);
int b2_space_coords(const b2_space* sp, int axis, double* x_host /* n values */);
/* diagnostic, no reference counterpart: the lane-kernel layout chosen for one pass orientation when the space was created
 * (orient 0: lanes along axis 1, orient 1: lanes along axis 0).  out8 = {E points per thread, LN lanes per CTA, TPL threads
 * per lane, fast (compile-time-geometry instance), CHW tiles per sub-chunk, sub-chunks per lane, threads per CTA, shared bytes} */
int b2_space_lane_layout(const b2_space* sp, int orient, int* out8);

/* ---- device arrays (the `Array2<T>` values that flow between Field and Solve calls) ---- */
int b2_array_create(b2_space* sp, int shape_kind, b2_array** out);
int b2_array_destroy(b2_array* a);
/* slab decomposition (funspace Decomp2d y-pencil, src/field_mpi.rs:130-134): axis 0 is split in
 * contiguous blocks of P0/nranks rows (P0 = rows padded to 4*nranks); with one rank this is the
 * whole array.  Host buffers of set/get hold exactly these rows (modes for complex arrays). */
int b2_array_local_rows(const b2_array* a, int* row_start, int* row_count);
int b2_array_sumsq_local(const b2_array* a, double* out);
int b2_array_set_host(b2_array* a, const void* buf, size_t bytes);
int b2_array_get_host(const b2_array* a, void* buf, size_t bytes);
int b2_array_axpy(b2_array* y, double alpha, const b2_array* x); /* y += alpha x (same shape kind) */
/* diagnostics on the device (callback(): src/navier_stokes/functions.rs:146-233, src/field/average.rs:26-59, src/field_mpi/average.rs:15-61) */
int b2_field_array(b2_field* f, int which /* 0 = v, 1 = vhat */, b2_array** out /* borrowed */);
int b2_array_copy(b2_array* dst, const b2_array* src);                                            /* same padded shape */
int b2_array_combine(b2_array* dst, const b2_array* a, const b2_array* b, int op, double alpha);   /* 0: alpha a b; 1: alpha sqrt(a^2+b^2); 2: dst + alpha a b */
/* dx-weighted sums over this rank's rows of a real array: mode 0: out[0] = sum_ij w0[i] w1[j] a[i][j]; mode 1: out[j] = sum_i w0[i] a[i][j]
 * (w0: one weight per LOCAL row, w1 / out: one per column; the caller adds the ranks' partial sums -- all_gather_sum);
 * mode 2: out[i] = sum_j w1[j] a[i][j] for this rank's LOCAL rows i (average_axis(1); the caller concatenates the ranks' parts) */
int b2_array_weighted_sum(const b2_array* a, const double* w0_local, const double* w1, int mode, double* out);
int b2_array_norm2(const b2_array* a, double* out);              /* sqrt(sum |a|^2) of the GLOBAL array (collective over the ranks), functions.rs:24-35 */

/* ---- Field2 (src/field.rs:59-129) ---- */
int b2_field_create(b2_space* sp, b2_field** out);                    /* Field2::new */
int b2_field_destroy(b2_field* f);
int b2_field_set_v_host(b2_field* f, const void* buf, size_t bytes);  /* field.v  <- host */
int b2_field_get_v_host(const b2_field* f, void* buf, size_t bytes);
int b2_field_set_vhat_host(b2_field* f, const void* buf, size_t bytes);
int b2_field_get_vhat_host(const b2_field* f, void* buf, size_t bytes);
int b2_field_local_rows(const b2_field* f, int shape_kind, int* row_start, int* row_count);
int b2_forward(b2_field* f);                                          /* field.rs:103-105 */
int b2_backward(b2_field* f);                                         /* field.rs:108-110 */
int b2_to_ortho(const b2_field* f, b2_array* out /* ORTHO */);        /* field.rs:113-115 */
int b2_from_ortho(b2_field* f, const b2_array* in /* ORTHO */);       /* field.rs:118-123 */
int b2_gradient(const b2_field* f, int d0, int d1, const double* scale /* 2 values or NULL */,
                b2_array* out /* ORTHO */);                           /* field.rs:127-129 */
int b2_field_dealias(b2_field* f);   /* dealias(&mut field): 2/3 rule on vhat, src/navier_stokes/functions.rs:72-82 */

/* ---- solvers (src/solver.rs:59-97 `Solve::solve(input, output, axis)`) ---- */
/* HholtzAdi::new(&field, [c0, c1]), src/solver/hholtz_adi.rs:48-76 */
int b2_hholtz_adi_create(const b2_field* f, double c0, double c1, b2_solver** out);
/* Poisson::new(&field, [c0, c1]), src/solver/poisson.rs:54-94.  For a Chebyshev axis 0 the
 * eigendecomposition of src/solver/fdma_tensor.rs:117-129 is supplied by the host (LAPACK dgeev,
 * as the reference): lam[m0] sorted descending (already shifted by the 1e-10 singularity rule of
 * poisson.rs:84-86), fwd[m0*m0] = Q^-1 C0^-1, bwd[m0*m0] = Q, row-major.  NULL for a Fourier axis 0. */
int b2_poisson_create(const b2_field* f, double c0, double c1, const double* lam, const double* fwd,
                      const double* bwd, b2_solver** out);
/* Hholtz::new(&field, [c0, c1]), src/solver/hholtz.rs:66-101: (I - c D2) vhat = A f through the same FdmaTensor as
 * Poisson (laplacian = -c * mat_b, mass = mat_a, alpha = 1, no singularity shift); lam / fwd / bwd = eigendecomposition of
 * C0^-1 (-c0 B0) as for b2_poisson_create (NULL for a Fourier axis 0). */
int b2_hholtz_create(const b2_field* f, double c0, double c1, const double* lam, const double* fwd,
                     const double* bwd, b2_solver** out);
int b2_solver_destroy(b2_solver* s);
/* solver.solve(&input [ORTHO], &mut output [SPECTRAL], 0) */
int b2_solve(b2_solver* s, const b2_array* in, b2_array* out);
/* host-side ingredients so that the caller can run LAPACK on exactly the matrices of
 * src/field.rs:195-249: X = C0^-1 A0 is returned through its banded factors */
int b2_poisson_axis0_matrices(const b2_field* f, double c0, double* a0 /* m0*m0 */, double* cmat0 /* m0*m0 */);
/* same, host only (no GPU needed): kind0/n0 of the pseudo-pressure axis-0 base */
int b2_host_poisson_matrices(int kind0, int n0, double c0, double* a0, double* cmat0);

/* ---- Navier2D (src/navier_stokes/navier.rs:215-466; MPI twin src/navier_stokes_mpi/navier.rs) ---- */
int b2_navier2d_create(b2_ctx* ctx, int nx, int ny, double ra, double pr, double dt, double aspect,
                       const char* bc /* "rbc" or "hc" */, int periodic, const double* lam, const double* fwd,
                       const double* bwd, b2_navier** out);
int b2_navier_destroy(b2_navier* nav);
/* which: 0 temp, 1 velx, 2 vely, 3 pres, 4 pseu, 5 tempbc */
int b2_navier_field(b2_navier* nav, int which, b2_field** out);
int b2_navier_update(b2_navier* nav, int nsteps);            /* Integrate::update, navier.rs:438-466 */
int b2_navier_div_norm(b2_navier* nav, double* out);         /* navier_eq.rs:32-49 (exit() NaN guard); the global norm on every rank */
int b2_navier_get_time(const b2_navier* nav, double* t);
int b2_navier_set_time(b2_navier* nav, double t);            /* restart: `self.time = read_scalar(.., "time")`, navier_io.rs:30 */
int b2_navier_set_mode(b2_navier* nav, int mode);            /* bit0: fused schedule (default on); bit1: no CUDA-graph replay */
/* schedule facts for bench.py: out[8] = {parity-block GEMMs, P0, P1, m0, ce, co, parallel branches, launches per step} */
int b2_navier_info(const b2_navier* nv, long long* out8);
int b2_navier_launch_count(const b2_navier* nav, long long* kernels_per_step);
int b2_navier_poisson_matrices(b2_navier* nav, double* a0, double* cmat0, int* m0);

#ifdef __cplusplus
}
#endif
#endif
