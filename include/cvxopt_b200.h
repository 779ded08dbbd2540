/*
 * cvxopt_b200 — C ABI of the B200-native KKT hot path of CVXOPT's cone solvers.
 *
 * Every entry point below is what a CVXOPT-side binding for this path would
 * bind (ctypes / CPython C-API; see INTEGRATION.md).  Plain pointers and sizes
 * only; no torch / Python types.  All matrices are fp64, column-major (the
 * layout of cvxopt's `matrix`, reference src/C/cvxopt.h:48-56), all index
 * arguments are 0-based element counts.
 *
 * Cone layout of every "cone vector" (reference src/python/coneprog.py:79-96):
 *   [ mnl nonlinear | ml 'l' | q[0] .. q[nq-1] 'q' blocks | s[0]^2 .. 's' blocks ]
 *   cdim      = mnl + ml + sum q + sum s^2        (unpacked, 's' blocks full col-major)
 *   cdim_pckd = mnl + ml + sum q + sum s(s+1)/2   (packed lower, off-diag * sqrt 2)
 *
 * Return codes (all int-returning functions):
 *    0   success
 *   >0   LAPACK-style `info`: leading minor of that order is not positive
 *        definite (the reference raises ArithmeticError for this,
 *        src/C/lapack.c:32-34) — Python layer raises ArithmeticError
 *   <0   CVXB_E_* below (bad argument / CUDA failure); cvxb_last_error() has text
 */
#ifndef CVXOPT_B200_H
#define CVXOPT_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define CVXB_E_ARG     (-1)   /* invalid argument (ValueError in the reference, misc.h:78-110) */
#define CVXB_E_CUDA    (-2)   /* CUDA runtime error */
#define CVXB_E_NOMEM   (-3)   /* allocation failure */
#define CVXB_E_NOGPU   (-4)   /* no usable sm_100 device: the product path has NO CPU fallback */
#define CVXB_E_UNSUP   (-5)   /* valid in the reference but not built on the device */

/* memory space of the pointers handed to a call */
#define CVXB_HOST   0
#define CVXB_DEVICE 1

typedef struct cvxb_kkt cvxb_kkt;     /* opaque: one kkt_chol factory instance  */
typedef struct cvxb_batch cvxb_batch; /* opaque: batch of independent dense QPs */

/* cone dimensions: mirror of the reference `dims` dict + mnl */
typedef struct {
    int mnl;          /* nonlinear rows (cvxprog), 0 for conelp/coneqp            */
    int ml;           /* dims['l']                                                 */
    int nq;           /* len(dims['q'])                                            */
    const int *q;     /* dims['q'][k]                                              */
    int ns;           /* len(dims['s'])                                            */
    const int *s;     /* dims['s'][k]                                              */
} cvxb_dims;

/* Nesterov-Todd scaling: flat mirror of the reference `W` dict
 * (src/python/coneprog.py:327-334, src/python/misc.py:45-56) */
typedef struct {
    const double *dnl, *dnli;   /* mnl each (may be NULL when mnl == 0)           */
    const double *d, *di;       /* ml each                                         */
    const double *v;            /* W['v'][0] | W['v'][1] | ...   (sum q)           */
    const double *beta;         /* nq                                              */
    const double *r, *rti;      /* W['r'][k] / W['rti'][k], s[k] x s[k] col-major,
                                   concatenated (sum s^2)                          */
} cvxb_scaling;

/* ---- library / device ---------------------------------------------------- */
const char *cvxb_last_error(void);
int  cvxb_device_count(void);                 /* sm_100 devices visible            */
int  cvxb_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
unsigned long long cvxb_launch_count(void);
/* cudaMalloc/cudaFree/cudaMemcpy shims so a ctypes-only host needs no CUDA binding */
int  cvxb_malloc(void **dptr, unsigned long long bytes);
int  cvxb_free(void *dptr);
int  cvxb_memcpy_h2d(void *dst, const void *src, unsigned long long bytes);
int  cvxb_memcpy_d2h(void *dst, const void *src, unsigned long long bytes);
int  cvxb_sync(void);

/* ---- kkt_chol factory:  replaces misc.kkt_chol(G, dims, A, mnl)
 *      reference src/python/misc.py:1213-1255.
 * G is cdim x n (rows mnl.. hold G; the mnl leading rows are Df, given per
 * factor call).  G is uploaded ONCE and stays resident in HBM.
 * space = CVXB_HOST: G/A are host pointers (copied); CVXB_DEVICE: device
 * pointers that are ADOPTED without copy (caller keeps them alive). */
int cvxb_kkt_create(cvxb_kkt **out, int n, int p, const cvxb_dims *dims,
                    const double *G, int ldg, const double *A, int lda,
                    int space, int device);
void cvxb_kkt_destroy(cvxb_kkt *k);

/* Factorisation route of this factory, chosen once right after cvxb_kkt_create:
 *   0  Cholesky of the reduced system           misc.kkt_chol / kkt_chol2   (misc.py:1213, :1352)  [default]
 *   1  QR:  A' = [Q1 Q2][R1; 0] (Householder, once), W^{-T} G Q2 = Q3 R3 per factor (Cholesky-QR with
 *      re-orthogonalisation, shifted when ill-conditioned)        misc.kkt_qr   (misc.py:1570-1699)
 *   2  LDL' with Bunch-Kaufman pivoting of the 2x2 system [H + Gs'Gs, A'; A, 0]   misc.kkt_ldl2 (misc.py:1128-1210);
 *      kktreg != 0 adds the reference's regularisation (misc.py:1096-1098 convention) to the diagonal.
 * Route 1 accepts no H / Df (zero (1,1) block, conelp). */
int cvxb_kkt_set_method(cvxb_kkt *k, int method, double kktreg);

/* Start a new solver run on the same factory (G, A, H stay resident): forgets the first-factorisation state
 * ("S singular on the first call -> S + A'A for the rest of the run", misc.py:1433-1447). */
int cvxb_kkt_reset(cvxb_kkt *k);

/* Make H (n x n, lower triangle significant) resident; later factor calls with
 * H == NULL and use_resident_H=1 add it.  coneqp passes the same P every
 * iteration (coneprog.py:1980-1981) — this avoids re-uploading n^2 doubles. */
int cvxb_kkt_set_H(cvxb_kkt *k, const double *H, int ldh, int space);

/* factor: replaces the closure `factor(W, H, Df)`  misc.py:1257-1282
 *   Gs = pack(W^{-T} [Df; G]);  K = Gs'Gs + H (lower);  K = L L'
 * W pointers live in `space`.  H/Df may be NULL.  use_resident_H: add the
 * matrix given to cvxb_kkt_set_H.  Returns info>0 on a non-positive pivot. */
int cvxb_kkt_factor(cvxb_kkt *k, const cvxb_scaling *W, const double *H, int ldh,
                    const double *Df, int lddf, int use_resident_H, int space);

/* solve: replaces the closure `solve(x, y, z)`  misc.py:1284-1345.
 * In place: (bx, by, bz) -> (ux, uy, W*uz).  x: n, y: p, z: cdim. */
int cvxb_kkt_solve(cvxb_kkt *k, double *x, double *y, double *z, int space);

/* read back pieces for tests: the Cholesky factor (n x n lower) */
int cvxb_kkt_get_L(cvxb_kkt *k, double *L_host, int ldl);
/* timing of the last factor/solve in ms (CUDA events on the library stream) */
int cvxb_kkt_last_ms(cvxb_kkt *k, double *factor_ms, double *solve_ms);
/* bracket a timed region with CUDA events on the library's launch stream (bench.py):
 * start records an event; stop records, synchronises and returns the elapsed ms */
int cvxb_kkt_timer_start(cvxb_kkt *k);
int cvxb_kkt_timer_stop(cvxb_kkt *k, double *ms);
/* debug (env CVXB_TRACE=1): globaltimer timeline of the last Cholesky, 8 values per block step:
 * {diag, trsm, next-column update, bulk update} x {start, end} in ns */
int cvxb_kkt_trace(cvxb_kkt *k, unsigned long long *out, int nsteps);
/* per-kernel-class CUDA-event breakdown of the last factor (syrk, potrf, scale) */
int cvxb_kkt_last_breakdown(cvxb_kkt *k, double *ms3);
/* which kernel computed the 'l'-row SYRK of the last factor: 0 none (ml == 0), 1 fp64 DMMA
 * (mma.sync.m8n8k4.f64), 2 int8 slices on tcgen05.mma kind::i8 (large problems; CVXB_OZAKI=0 disables,
 * falls back to 1 when the slice workspace does not fit in device memory) */
int cvxb_kkt_syrk_path(cvxb_kkt *k);
/* int8-slice path only: CUDA-event time of the MMA launches of the last factor's SYRK, without the two slicing kernels
 * (0 on the DMMA path); bench.py's roofline line divides the int8 operations by this */
int cvxb_kkt_syrk_mma_ms(cvxb_kkt *k, double *ms);
/* QR route: Cholesky-QR passes of the last factor: 2 (plain, re-orthogonalised) or 3 (shifted, ill-conditioned) */
int cvxb_kkt_qr_passes(cvxb_kkt *k);

/* device-resident G / P operators for the function-valued G(x,y,alpha,beta,trans)
 * / P(x,y,alpha,beta) protocol of coneprog (coneprog.py:1682-1711):
 *   y := alpha*G*x + beta*y  (trans 'N')   or   y := alpha*G'*x + beta*y ('T')
 *   y := alpha*H*x + beta*y  (H symmetric, lower stored) */
int cvxb_kkt_gemv_G(cvxb_kkt *k, const double *x, double *y, double alpha, double beta,
                    int trans, int space);
int cvxb_kkt_symv_H(cvxb_kkt *k, const double *x, double *y, double alpha, double beta,
                    int space);
/* y := alpha*A*x + beta*y ('N') or alpha*A'*x + beta*y ('T') on the resident equality-constraint
 * matrix: the function-valued A(x, y, alpha, beta, trans) protocol (coneprog.py:1682-1711) */
int cvxb_kkt_gemv_A(cvxb_kkt *k, const double *x, double *y, double alpha, double beta,
                    int trans, int space);

/* ---- cone algebra: mirror of src/C/misc_solvers.c (12 entry points,
 * misc_solvers.c:1155-1173).  x is xr x xc column-major with leading
 * dimension xr; everything in place as in the reference. */
int cvxb_scale(double *x, int xr, int xc, const cvxb_dims *dims, const cvxb_scaling *W,
               int trans /*'N'|'T'*/, int inverse /*'N'|'I'*/, int space); /* misc_solvers.c:85  */
int cvxb_scale2(const double *lmbda, double *x, const cvxb_dims *dims, int inverse,
                int space);                                                  /* :256 */
int cvxb_pack(const double *x, double *y, const cvxb_dims *dims, int space); /* :412 */
int cvxb_pack2(double *x, int xr, int xc, const cvxb_dims *dims, int space); /* :476 */
int cvxb_unpack(const double *x, double *y, const cvxb_dims *dims, int space); /* :552 */
int cvxb_symm(double *x, int n, int space);                                  /* :610 */
int cvxb_sprod(double *x, const double *y, const cvxb_dims *dims, int diag, int space);  /* :634 */
int cvxb_sinv(double *x, const double *y, const cvxb_dims *dims, int space); /* :775 */
int cvxb_trisc(double *x, const cvxb_dims *dims, int space);                 /* :887 */
int cvxb_triusc(double *x, const cvxb_dims *dims, int space);                /* :940 */
int cvxb_sdot(const double *x, const double *y, const cvxb_dims *dims, double *result,
              int space);                                                    /* :991 */
/* sigma == NULL: x is read only.  sigma != NULL (sum of the 's' orders): the eigenvalues of every 's'
 * block go to sigma (ascending) and its eigenvectors overwrite the block of x (:1132-1136).
 * Returns 1 if the eigensolver does not converge (non-finite input). */
int cvxb_max_step(double *x, const cvxb_dims *dims, double *sigma, double *result,
                  int space);                                                /* :1052 */

/* ---- Nesterov-Todd scaling itself: misc.compute_scaling (src/python/misc.py:250-419) and
 * misc.update_scaling (:422-634) for every cone type.  `W` points at WRITABLE arrays laid out as in
 * cvxb_scaling (the const qualifiers of that struct are cast away for these two calls): compute_scaling fills
 * them, update_scaling updates them in place together with lmbda; update_scaling also overwrites s and z the
 * way the reference does.  lmbda has mnl + ml + sum q + sum s entries.  's' blocks: Cholesky + one-sided Jacobi
 * SVD on the device in place of lapack.potrf / lapack.gesvd; singular values in descending order.
 * Returns info > 0 if an 's' block is not positive definite (ArithmeticError in the reference). */
int cvxb_compute_scaling(const double *s, const double *z, double *lmbda, const cvxb_dims *dims,
                         const cvxb_scaling *W, int space);
int cvxb_update_scaling(const cvxb_scaling *W, double *lmbda, double *s, double *z,
                        const cvxb_dims *dims, int space);

/* ---- dense building blocks (the BLAS/LAPACK calls of the path, device pointers):
 * blas.syrk(trans='T') blas.c:3039 fused with the 'l' row scaling;
 * lapack.potrf lapack.c:1471; lapack.potrs lapack.c:1553. */
int cvxb_syrk_scaled(int n, int k, const double *A, int lda, const double *rowscale,
                     const double *H, int ldh, double *C, int ldc, int device);
/* The same SYRK, C(lower) = A' diag(d)^2 A + H, computed on the int8 tensor path by error-free
 * slicing (Ozaki scheme, `slices` = 1..9 radix-2^7 digits per entry; 9 reproduces fp64).  Note d, not
 * d^2 as in cvxb_syrk_scaled.  cvxb_kkt_factor uses it for large 'l' blocks (CVXB_OZAKI=0 disables).
 * blas.syrk blas.c:3039. */
int cvxb_syrk_scaled_i8(int n, int k, const double *A, int lda, const double *d, const double *H,
                        int ldh, double *C, int ldc, int slices, int device);
/* work_inv: 2 * ceil(n/128) * 128*128 doubles — receives the inverses (and their
 * transposes) of the 128x128 diagonal blocks of L, consumed by cvxb_potrs */
int cvxb_potrf(int n, double *A, int lda, double *work_inv, int device);
int cvxb_potrs(int n, const double *L, int ldl, const double *inv, double *b, int device);
/* plain C = alpha * op(A) op(B) + beta*C on the DMMA kernel (tests / 's' congruence) */
int cvxb_gemm(int transa, int transb, int m, int n, int k, double alpha, const double *A,
              int lda, const double *B, int ldb, double beta, double *C, int ldc, int device);

/* ---- batch of independent dense QPs (BASELINE config 4): one problem per
 * CTA-group, lock-step primal-dual IPM fully on device (oracle: a Python loop
 * over solvers.qp).  Problems are  min 1/2 x'P x + q'x  s.t.  G x <= h, A x = b,
 * A with p rows (0 <= p <= n; p > 0 needs m > 0).  With p > 0 every problem
 * follows coneqp with kktsolver='chol2' (solvers.qp(P, q, G, h, A, b)).
 * cvxb_batch_create is cvxb_batch_create_eq with p = 0.
 * cvxb_batch_create_cones: the inequalities are the cone dims = {'l': ml, 'q': [q[0] .. q[nq-1]]}, the same for
 * every problem: rows of G and h are ml linear rows, then the second-order cones in order (m = ml + sum q, each
 * q[k] >= 1).  Every problem follows coneqp(P, q, G, h, dims[, A, b]) with the reference's default options.
 * cvxb_batch_create_eq(.., m, p, ..) is cvxb_batch_create_cones with ml = m, nq = 0. */
int cvxb_batch_create(cvxb_batch **out, int nprob, int n, int m, int device);
int cvxb_batch_create_eq(cvxb_batch **out, int nprob, int n, int m, int p, int device);
int cvxb_batch_create_cones(cvxb_batch **out, int nprob, int n, int ml, int nq, const int *q, int p, int device);
void cvxb_batch_destroy(cvxb_batch *b);
/* P: nprob x (n x n, ld n); q: nprob x n; G: nprob x (m x n column-major, ld m); h: nprob x m */
int cvxb_batch_load(cvxb_batch *b, const double *P, const double *q, const double *G,
                    const double *h, int space);
/* A: nprob x (p x n column-major, ld p); bvec: nprob x p.  Required after every
 * cvxb_batch_load when p > 0 (a no-op when p = 0). */
int cvxb_batch_load_eq(cvxb_batch *b, const double *A, const double *bvec, int space);
int cvxb_batch_solve(cvxb_batch *b, int maxiters, double abstol, double reltol, double feastol);
/* the same with coneqp's options['refinement']: steps of iterative refinement per Newton solve; a negative value
 * is the reference's default (1 with 'q' cones, else 0), which is what cvxb_batch_solve uses */
int cvxb_batch_solve_ref(cvxb_batch *b, int maxiters, double abstol, double reltol, double feastol,
                         int refinement);
/* status: 1 optimal, 2 maximum iterations reached, 3 singular KKT matrix ('unknown' in the
 * reference for 2 and 3).  x/s/z may be device pointers (space), scalars go to host memory. */
int cvxb_batch_results(cvxb_batch *b, double *x, double *s, double *z, int *status,
                       int *iters, double *pobj, double *dobj, int space);
/* y: nprob x p multipliers of A x = b (host or device memory, space) */
int cvxb_batch_results_y(cvxb_batch *b, double *y, int space);
/* flags (host, nprob): 1 where S = P + G'W^-1 W^-T G was singular at the starting point,
 * so that S + A'A was factored instead (the reference's kkt_chol2 'singular' branch) */
int cvxb_batch_singular(cvxb_batch *b, int *flags);
/* ms[3]: time of the last solve's factorisations by phase: S (SYRK + Cholesky),
 * L^{-1} A' (TRSM), A S^{-1} A' (SYRK + Cholesky).  Only for a batch created with
 * CVXB_BATCH_PHASE_MS=1, which synchronises after every phase. */
int cvxb_batch_phase_ms(cvxb_batch *b, double *ms);
/* ms[2]: the part of phase S spent on the 'q' rows: Gs_q = W^-T G_q, and the GEMM K += Gs_q' Gs_q (same batches) */
int cvxb_batch_phase_ms_cones(cvxb_batch *b, double *ms);
/* CUDA-event time of the last cvxb_batch_solve and the number of lock-step iterations run */
int cvxb_batch_stats(cvxb_batch *b, double *solve_ms, int *iterations);
/* kernel of the factorisations' SYRK in the last solve: 1 fp64 DMMA, 2 int8 slices (as cvxb_kkt_syrk_path) */
int cvxb_batch_syrk_path(cvxb_batch *b);

#ifdef __cplusplus
}
#endif
#endif /* CVXOPT_B200_H */
