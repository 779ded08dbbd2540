// Internal definition of the KKT factory handle shared by kkt_api.cu (Cholesky route, misc.kkt_chol / kkt_chol2),
// kkt_qr.cu (misc.kkt_qr) and kkt_ldl.cu (misc.kkt_ldl2).
#pragma once
#include "cone.cuh"

using cvxb::ConeLayout;
using cvxb::DevScaling;
using cvxb::CholWork;

struct cvxb_kkt {
    int device = 0;
    int n = 0, p = 0;
    ConeLayout cone;
    const double *G = nullptr;   // cdim x n, rows [mnl, cdim) hold G (rows [0,mnl) belong to Df)
    long long ldg = 0;
    bool own_G = false;
    double *Hres = nullptr;      // resident H (symmetrised), or null
    double *Hbuf = nullptr;      // per-call H upload buffer (lazy)
    double *Kmat = nullptr;      // n x n: normal equations, then its Cholesky factor (lower)
    double *inv = nullptr;       // inverses of the diagonal blocks of L
    double *Gs = nullptr;        // scaled+packed rows that are not 'l': [mnl | q | s packed] x n
    long long ldgs = 0;
    int nrest = 0;
    double *Gunp = nullptr;      // unpacked scaled 's' rows (sums2 x n) — only when ns > 0
    double *Dfbuf = nullptr;     // mnl x n upload buffer
    // equality constraints (p > 0), kkt_chol2-style elimination (reference misc.py:1464-1472):
    double *Aeq = nullptr;       // p x n (ld lda_eq)
    long long lda_eq = 0;
    double *Asct = nullptr;      // n x p: L^{-1} A'
    long long ldas = 0;
    double *Kp = nullptr;        // p x p: Asct' Asct, then its Cholesky factor
    long long ldkp = 0;
    double *invp = nullptr;      // diagonal-block inverses of chol(Kp)
    double *yd = nullptr;        // p
    bool singular = false;       // first factorisation failed -> S += A'A from then on (misc.py:1433-1447)
    bool first_factor = true;
    DevScaling W;
    double *bzp = nullptr, *zin = nullptr, *zt = nullptr, *xv = nullptr, *yv = nullptr;
    double *gemv_ws = nullptr;
    double *swork = nullptr;
    size_t swork_doubles = 0;
    CholWork cw;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr, e3 = nullptr, t0 = nullptr, t1 = nullptr;
    cudaEvent_t m0 = nullptr, m1 = nullptr;      // around the MMA launches of the int8-slice SYRK
    double mma_ms = 0.0;
    double factor_ms = 0, solve_ms = 0, br[3] = {0, 0, 0};
    bool factored = false;
    // SYRK of the 'l' rows on the int8 tensor path (ozaki_syrk.cu): 0 off (DMMA kernel), 1 for large
    // problems (where it measured faster), 2 always.  CVXB_OZAKI=0/1/2 read at create; unset = 1.
    int i8_mode = 1;
    void *oz_work = nullptr;
    size_t oz_bytes = 0;
    int syrk_path = 0;           // kernel of the last factor's 'l'-row SYRK: 0 none, 1 fp64 DMMA, 2 int8 slices
    // factorisation route: 0 Cholesky of the reduced system (kkt_chol / kkt_chol2), 1 QR (kkt_qr), 2 LDL' of the
    // 2x2 system (kkt_ldl2).  Set once after create (cvxb_kkt_set_method); state of routes 1/2 lives in `ext`.
    int method = 0;
    void *ext = nullptr;
    void (*ext_destroy)(void *) = nullptr;
};


namespace cvxb {
int upload_matrix(double *dst, long long ldd, const double *src, long long lds, int rows, int cols, int space,
                  cudaStream_t st);
int xfer_vec(double *dst, const double *src, size_t n, int space, bool to_device, cudaStream_t st);
inline long long kkt_ldk(const cvxb_kkt *k) { long long l = (k->n + 1) & ~1; return l > 2 ? l : 2; }
// B := L^{-1} B for the n x n Cholesky factor L (lower, ld ldl) with its diagonal-block inverses `inv`
// (potrf_lower's output); B is n x ncols (ld ldb), updated in place by blocked forward substitution (DMMA GEMMs).
// Batched (blockIdx.z of every GEMM): problem b uses L + b*sL, inv + b*sInv, B + b*sB.
int trsm_lower_left(int n, const double *L, long long ldl, const double *inv, double *B, long long ldb, int ncols,
                    cudaStream_t st, int batch = 1, long long sL = 0, long long sInv = 0, long long sB = 0);
int kkt_pack_bz(cvxb_kkt *k, const double *zd);      // k->bzp := pack(W^{-T} bz)
int kkt_unpack_z(cvxb_kkt *k, double *zd);           // z := unpack(k->bzp)
// route-specific factor / solve (kkt_qr.cu, kkt_ldl.cu)
int kkt_qr_factor(cvxb_kkt *k, const cvxb_scaling *W, int space);
int kkt_qr_solve(cvxb_kkt *k, double *x, double *y, double *z, int space);
int kkt_qr_setup(cvxb_kkt *k);
int kkt_qr_passes(const cvxb_kkt *k);
// LDL' route: Kmat holds S (lower) on entry of factor; info (k->cw.d_info) = first exactly-zero pivot, 1-based
int kkt_ldl_factor(cvxb_kkt *k);
int kkt_ldl_solve(cvxb_kkt *k, double *xd, double *yd);        // device vectors, in place
int kkt_ldl_setup(cvxb_kkt *k, double kktreg);
}  // namespace cvxb
