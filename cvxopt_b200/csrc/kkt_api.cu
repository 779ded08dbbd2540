// C ABI of the KKT hot path (see include/cvxopt_b200.h).
//
// cvxb_kkt mirrors the closure chain of the reference's misc.kkt_chol
// (src/python/misc.py:1213-1349):  create == kkt_chol(G, dims, A),
// factor == factor(W, H, Df), solve == solve(x, y, z).  G (and optionally H) are
// uploaded once and stay resident in HBM; per factor only the O(cdim) scaling
// parameters cross PCIe, per solve only the right-hand side / solution.
#include "cone.cuh"
#include <cstdlib>
#include <cstdarg>
#include <mutex>

#include <map>
#include <unordered_map>
#include <mutex>
#include <iterator>
#include <cstdlib>

namespace cvxb {

static thread_local std::string g_err;
std::atomic<unsigned long long> g_launches{0};


// ---- scratch-buffer cache (common.cuh) ----
namespace {
struct TmpCache {
    std::mutex mu;
    std::multimap<size_t, void *> free_[64];          // per device: block size -> pointer
    std::unordered_map<void *, std::pair<size_t, int>> live;   // handed-out blocks: size, device
    size_t cached = 0, cap = 0;
    bool cap_set = false;
};
TmpCache &tmpc() { static TmpCache *c = new TmpCache; return *c; }   // never destroyed: frees may come after main()
size_t tmp_round(size_t b) { return b <= 4096 ? 4096 : (b + 65535) & ~(size_t)65535; }
void tmp_drop_all_locked(TmpCache &c) {
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < 64; ++d) {
        if (c.free_[d].empty()) continue;
        cudaSetDevice(d);
        for (auto &kv : c.free_[d]) cudaFree(kv.second);
        c.free_[d].clear();
    }
    cudaSetDevice(cur);
    c.cached = 0;
}
}  // namespace

cudaError_t tmp_malloc_bytes(void **p, size_t bytes) {
    TmpCache &c = tmpc();
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const size_t want = tmp_round(bytes ? bytes : 1);
    std::lock_guard<std::mutex> g(c.mu);
    auto &fl = c.free_[dev & 63];
    auto it = fl.lower_bound(want);
    if (it != fl.end() && it->first <= want + want / 4) {
        *p = it->second;
        c.live[*p] = {it->first, dev};
        c.cached -= it->first;
        fl.erase(it);
        return cudaSuccess;
    }
    e = cudaMalloc(p, want);
    if (e != cudaSuccess) {                       // out of memory: give the cached blocks back and retry once
        cudaGetLastError();
        tmp_drop_all_locked(c);
        e = cudaMalloc(p, want);
        if (e != cudaSuccess) return e;
    }
    c.live[*p] = {want, dev};
    return cudaSuccess;
}

void tmp_free(void *p) {
    if (!p) return;
    TmpCache &c = tmpc();
    std::lock_guard<std::mutex> g(c.mu);
    auto it = c.live.find(p);
    if (it == c.live.end()) { cudaFree(p); return; }          // not ours (defensive)
    const size_t sz = it->second.first;
    const int dev = it->second.second;
    c.live.erase(it);
    if (!c.cap_set) {
        const char *e = getenv("CVXB_TMP_CACHE_MB");
        c.cap = (size_t)(e ? atoll(e) : 4096) << 20;
        c.cap_set = true;
    }
    if (sz > c.cap) { cudaFree(p); return; }
    while (c.cached + sz > c.cap) {                           // evict the largest cached blocks first
        size_t best = 0; int bd = -1;
        for (int d = 0; d < 64; ++d)
            if (!c.free_[d].empty() && c.free_[d].rbegin()->first >= best) { best = c.free_[d].rbegin()->first; bd = d; }
        if (bd < 0) break;
        auto last = std::prev(c.free_[bd].end());
        int cur = 0; cudaGetDevice(&cur);
        if (cur != bd) cudaSetDevice(bd);
        cudaFree(last->second);
        if (cur != bd) cudaSetDevice(cur);
        c.cached -= last->first;
        c.free_[bd].erase(last);
    }
    c.free_[dev & 63].emplace(sz, p);
    c.cached += sz;
}

void tmp_cache_release() {
    TmpCache &c = tmpc();
    std::lock_guard<std::mutex> g(c.mu);
    tmp_drop_all_locked(c);
}

void set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

static int check_device(int device) {
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s): cvxopt_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return CVXB_E_NOGPU;
    }
    if (device < 0 || device >= cnt) {
        set_error("device %d out of range (%d visible)", device, cnt);
        return CVXB_E_ARG;
    }
    cudaDeviceProp prop;
    CVXB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device,
                  prop.major, prop.minor);
        return CVXB_E_NOGPU;
    }
    CVXB_CUDA(cudaSetDevice(device));
    return 0;
}

}  // namespace cvxb

using namespace cvxb;

#include "kkt_internal.cuh"

namespace cvxb {

int upload_matrix(double *dst, long long ldd, const double *src, long long lds, int rows, int cols,
                  int space, cudaStream_t st) {
    if (rows <= 0 || cols <= 0) return 0;
    cudaMemcpyKind kind = (space == CVXB_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CVXB_CUDA(cudaMemcpy2DAsync(dst, ldd * sizeof(double), src, lds * sizeof(double),
                                (size_t)rows * sizeof(double), cols, kind, st));
    return 0;
}

int xfer_vec(double *dst, const double *src, size_t n, int space, bool to_device, cudaStream_t st) {
    if (n == 0) return 0;
    cudaMemcpyKind kind = (space == CVXB_DEVICE) ? cudaMemcpyDeviceToDevice
                          : (to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost);
    CVXB_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), kind, st));
    return 0;
}

// bzp := pack(W^{-T} bz)                                       (misc.py:1306-1307, :1626-1627)
int kkt_pack_bz(cvxb_kkt *k, const double *zd) {
    const ConeLayout &c = k->cone;
    cudaStream_t st = k->st;
    const int nlq = c.mnl + c.ml + c.sumq;
    if (c.mnl > 0) CVXB_TRY(scale_rows(zd, c.cdim, k->bzp, c.cdim, c.mnl, 1, k->W.dnli, st));
    if (c.ml > 0)
        CVXB_TRY(scale_rows(zd + c.mnl, c.cdim, k->bzp + c.mnl, c.cdim, c.ml, 1, k->W.di, st));
    if (c.nq > 0)
        CVXB_TRY(scale_q(c, k->W, zd + c.mnl + c.ml, c.cdim, k->bzp + c.mnl + c.ml, c.cdim, 1, true, st));
    if (c.ns > 0) {
        CVXB_TRY(scale_s(c, k->W, zd + nlq, c.cdim, k->zt + nlq, c.cdim, 1, 'T', 'I', k->swork,
                         k->swork_doubles, st));
        CVXB_TRY(pack_s(c, k->zt + nlq, c.cdim, k->bzp + nlq, c.cdim, 1, true, st));
    }
    return 0;
}

// z := unpack(bzp)                                             (misc.py:1345, :1697)
int kkt_unpack_z(cvxb_kkt *k, double *zd) {
    const ConeLayout &c = k->cone;
    cudaStream_t st = k->st;
    const int nlq = c.mnl + c.ml + c.sumq;
    if (nlq > 0)
        CVXB_CUDA(cudaMemcpyAsync(zd, k->bzp, (size_t)nlq * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (c.ns > 0) CVXB_TRY(unpack_s(c, k->bzp + nlq, c.cdim, zd + nlq, c.cdim, 1, st));
    return 0;
}

int trsm_lower_left(int n, const double *L, long long ldl, const double *inv, double *B, long long ldb, int ncols,
                    cudaStream_t st, int batch, long long sL, long long sInv, long long sB) {
    if (n <= 0 || ncols <= 0 || batch <= 0) return 0;
    const int nblk = (n + NB - 1) / NB;
    for (int jb = 0; jb < nblk; ++jb) {
        const int j = jb * NB;
        const int wj = (n - j < NB) ? (n - j) : NB;
        const int mrem = n - j - wj;
        double *Bj = B + j;
        {   // X_j = inv_jj * B_j   (in place: one tile row, every tile owns its columns)
            GemmDesc g;
            g.M = wj; g.N = ncols; g.K = wj;
            g.X = inv + (long long)jb * NB * NB; g.ldx = NB; g.x_kmajor = false;
            g.Y = Bj; g.ldy = (int)ldb; g.y_kmajor = true;
            g.C = Bj; g.ldc = (int)ldb;
            g.batch = batch; g.sX = sInv; g.sY = sB; g.sC = sB;
            CVXB_TRY(dmma_gemm(g, st));
        }
        if (mrem > 0) {   // B[j+1:, :] -= L[j+1:, j] X_j
            GemmDesc g;
            g.M = mrem; g.N = ncols; g.K = wj;
            g.X = L + (j + wj) + (long long)j * ldl; g.ldx = (int)ldl; g.x_kmajor = false;
            g.Y = Bj; g.ldy = (int)ldb; g.y_kmajor = true;
            g.D = Bj + wj; g.ldd = (int)ldb; g.C = Bj + wj; g.ldc = (int)ldb;
            g.alpha = -1.0; g.beta = 1.0;
            g.batch = batch; g.sX = sL; g.sY = sB; g.sD = sB; g.sC = sB;
            CVXB_TRY(dmma_gemm(g, st));
        }
    }
    return 0;
}

}  // namespace cvxb

extern "C" {

const char *cvxb_last_error(void) { return g_err.c_str(); }
int cvxb_version(void) { return 100; }
unsigned long long cvxb_launch_count(void) { return g_launches.load(); }

int cvxb_device_count(void) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < cnt; ++d) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) ++ok;
    }
    return ok;
}

int cvxb_malloc(void **dptr, unsigned long long bytes) {
    CVXB_CUDA(cudaMalloc(dptr, bytes ? bytes : 8));
    return 0;
}
int cvxb_free(void *dptr) { CVXB_CUDA(cudaFree(dptr)); return 0; }
int cvxb_memcpy_h2d(void *dst, const void *src, unsigned long long bytes) {
    CVXB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return 0;
}
int cvxb_memcpy_d2h(void *dst, const void *src, unsigned long long bytes) {
    CVXB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
}
int cvxb_sync(void) { CVXB_CUDA(cudaDeviceSynchronize()); return 0; }

// --------------------------------------------------------------------- create
int cvxb_kkt_create(cvxb_kkt **out, int n, int p, const cvxb_dims *dims, const double *G,
                    int ldg, const double *A, int lda, int space, int device) {
    if (!out) { set_error("kkt_create: out is NULL"); return CVXB_E_ARG; }
    *out = nullptr;
    if (n < 0 || p < 0) { set_error("kkt_create: negative size"); return CVXB_E_ARG; }
    if (p > 0 && (!A || lda < p)) { set_error("kkt_create: A must be p x n with lda >= p"); return CVXB_E_ARG; }
    if (p > n) { set_error("kkt_create: Rank(A) < p (p > n)"); return CVXB_E_ARG; }
    CVXB_TRY(check_device(device));
    cvxb_kkt *k = new cvxb_kkt();
    k->device = device; k->n = n; k->p = p;
    if (const char *e = getenv("CVXB_OZAKI")) k->i8_mode = (e[0] == '0') ? 0 : (e[0] == '2') ? 2 : 1;
    int rc = k->cone.init(dims);
    if (rc) { delete k; return rc; }
    const ConeLayout &c = k->cone;
    if (c.cdim > 0 && (!G || ldg < (c.cdim > 1 ? c.cdim : 1))) {
        set_error("kkt_create: G must be cdim x n with ldg >= cdim (cdim=%d, ldg=%d)", c.cdim, ldg);
        cvxb_kkt_destroy(k);
        return CVXB_E_ARG;
    }
    auto fail = [&](int r) { cvxb_kkt_destroy(k); return r; };
#define KTRY(expr) do { int _r = (expr); if (_r) return fail(_r); } while (0)
#define KCUDA(expr) do { cudaError_t _e = (expr); \
        /* out of memory: give the scratch-buffer cache (common.cuh) back to the driver and try once more */ \
        if (_e == cudaErrorMemoryAllocation) { cudaGetLastError(); tmp_cache_release(); _e = (expr); } \
        if (_e != cudaSuccess) { \
        set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
        return fail(_e == cudaErrorMemoryAllocation ? CVXB_E_NOMEM : CVXB_E_CUDA); } } while (0)
    KCUDA(cudaStreamCreateWithFlags(&k->st, cudaStreamNonBlocking));
    KCUDA(cudaEventCreate(&k->e0)); KCUDA(cudaEventCreate(&k->e1));
    KCUDA(cudaEventCreate(&k->e2)); KCUDA(cudaEventCreate(&k->e3));
    KCUDA(cudaEventCreate(&k->t0)); KCUDA(cudaEventCreate(&k->t1));
    KCUDA(cudaEventCreate(&k->m0)); KCUDA(cudaEventCreate(&k->m1));
    KTRY(chol_work_create(k->cw));
    const size_t nn = (size_t)(n > 0 ? n : 1);
    if (space == CVXB_DEVICE) {
        k->G = G; k->ldg = ldg; k->own_G = false;
    } else {
        double *g = nullptr;
        k->ldg = (c.cdim + 1) & ~1;     // even leading dimension: 16-byte aligned columns
        if (k->ldg < 2) k->ldg = 2;
        KCUDA(cudaMalloc(&g, (size_t)k->ldg * nn * sizeof(double)));
        k->G = g; k->own_G = true;
        KTRY(upload_matrix(g, k->ldg, G, ldg, c.cdim, n, CVXB_HOST, k->st));
    }
    const long long ldk = (n + 1) & ~1;
    KCUDA(cudaMalloc(&k->Kmat, (size_t)(ldk > 2 ? ldk : 2) * nn * sizeof(double)));
    const int nblk = (n + NB - 1) / NB + 1;
    KCUDA(cudaMalloc(&k->inv, (size_t)2 * nblk * NB * NB * sizeof(double)));   // inv + inv' blocks
    k->nrest = c.mnl + c.sumq + c.sump;
    if (k->nrest > 0) {
        k->ldgs = (k->nrest + 1) & ~1;
        KCUDA(cudaMalloc(&k->Gs, (size_t)k->ldgs * nn * sizeof(double)));
    }
    if (c.sums2 > 0) {
        KCUDA(cudaMalloc(&k->Gunp, (size_t)c.sums2 * nn * sizeof(double)));
        // workspace for the congruences: symmetric copies + intermediate, chunked over columns
        size_t per_col = (size_t)2 * c.maxs * c.maxs;
        size_t cols = (size_t)n < 1 ? 1 : (size_t)n;
        size_t want = per_col * cols;
        const size_t cap = (size_t)1 << 29;            // 4 GiB of doubles at most
        if (want > cap) want = (cap / per_col ? cap / per_col : 1) * per_col;
        k->swork_doubles = want;
        KCUDA(cudaMalloc(&k->swork, want * sizeof(double)));
    }
    if (c.mnl > 0) KCUDA(cudaMalloc(&k->Dfbuf, (size_t)c.mnl * nn * sizeof(double)));
    if (p > 0) {
        k->lda_eq = (p + 1) & ~1;
        k->ldas = (n + 1) & ~1;
        k->ldkp = (p + 1) & ~1;
        KCUDA(cudaMalloc(&k->Aeq, (size_t)k->lda_eq * nn * sizeof(double)));
        KCUDA(cudaMalloc(&k->Asct, (size_t)k->ldas * p * sizeof(double)));
        KCUDA(cudaMalloc(&k->Kp, (size_t)k->ldkp * p * sizeof(double)));
        KCUDA(cudaMalloc(&k->invp, (size_t)2 * ((p + NB - 1) / NB + 1) * NB * NB * sizeof(double)));
        KCUDA(cudaMalloc(&k->yd, (size_t)p * sizeof(double)));
        KTRY(upload_matrix(k->Aeq, k->lda_eq, A, lda, p, n, space, k->st));
    }
    KTRY(k->W.alloc(c));
    const size_t cd = (size_t)(c.cdim > 0 ? c.cdim : 1);
    KCUDA(cudaMalloc(&k->bzp, cd * sizeof(double)));
    KCUDA(cudaMalloc(&k->zin, cd * sizeof(double)));
    KCUDA(cudaMalloc(&k->zt, cd * sizeof(double)));
    KCUDA(cudaMalloc(&k->xv, nn * sizeof(double)));
    KCUDA(cudaMalloc(&k->yv, (cd > nn ? cd : nn) * sizeof(double)));
    {
        size_t w1 = cd * (size_t)gemv_n_chunks(n), w2 = nn * (size_t)gemv_n_chunks(p > 0 ? p : 1);
        const size_t w3 = (size_t)(p > 0 ? p : 1) * (size_t)gemv_n_chunks(n);      // A operator
        if (w3 > w1) w1 = w3;
        KCUDA(cudaMalloc(&k->gemv_ws, (w1 > w2 ? w1 : w2) * sizeof(double)));
    }
    KCUDA(cudaStreamSynchronize(k->st));
#undef KTRY
#undef KCUDA
    *out = k;
    return 0;
}

void cvxb_kkt_destroy(cvxb_kkt *k) {
    if (!k) return;
    cudaSetDevice(k->device);
    if (k->st) cudaStreamSynchronize(k->st);
    if (k->own_G && k->G) cudaFree(const_cast<double *>(k->G));
    double *bufs[] = {k->Aeq, k->Asct, k->Kp, k->invp, k->yd, k->Hres, k->Hbuf, k->Kmat, k->inv, k->Gs, k->Gunp, k->Dfbuf, k->bzp,
                      k->zin, k->zt, k->xv, k->yv, k->gemv_ws, k->swork};
    for (double *b : bufs) if (b) cudaFree(b);
    if (k->oz_work) cudaFree(k->oz_work);
    if (k->ext && k->ext_destroy) k->ext_destroy(k->ext);
    k->W.destroy();
    k->cone.destroy();
    chol_work_destroy(k->cw);
    cudaEvent_t evs[] = {k->e0, k->e1, k->e2, k->e3, k->t0, k->t1, k->m0, k->m1};
    for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
    if (k->st) cudaStreamDestroy(k->st);
    delete k;
}


int cvxb_kkt_set_method(cvxb_kkt *k, int method, double kktreg) {
    if (!k) { set_error("kkt is NULL"); return CVXB_E_ARG; }
    if (k->method != 0 || k->factored) { set_error("set_method: call once, right after create"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    if (method == 0) return 0;
    if (method == 1) { CVXB_TRY(kkt_qr_setup(k)); k->method = 1; return 0; }
    if (method == 2) { CVXB_TRY(kkt_ldl_setup(k, kktreg)); k->method = 2; return 0; }
    set_error("set_method: unknown method %d", method);
    return CVXB_E_ARG;
}

int cvxb_kkt_reset(cvxb_kkt *k) {
    if (!k) { set_error("kkt is NULL"); return CVXB_E_ARG; }
    // a new solver run on the same factory: the "S was singular on the first factorisation -> S + A'A from then
    // on" decision (misc.py:1433-1447) belongs to ONE run of the driver
    k->singular = false;
    k->first_factor = true;
    k->factored = false;
    return 0;
}

int cvxb_kkt_set_H(cvxb_kkt *k, const double *H, int ldh, int space) {
    if (!k) { set_error("kkt is NULL"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    if (!H) {
        if (k->Hres) cudaFree(k->Hres);
        k->Hres = nullptr;
        return 0;
    }
    if (ldh < (k->n > 1 ? k->n : 1)) { set_error("set_H: ldh < n"); return CVXB_E_ARG; }
    const long long ldk = kkt_ldk(k);
    if (!k->Hres) CVXB_CUDA(cudaMalloc(&k->Hres, (size_t)ldk * (k->n > 0 ? k->n : 1) * sizeof(double)));
    CVXB_TRY(upload_matrix(k->Hres, ldk, H, ldh, k->n, k->n, space, k->st));
    // only tril(H) is significant in the reference (misc.py:1276-1277); make the resident
    // copy fully symmetric so it also serves the P(x, y) operator
    CVXB_TRY(symmetrize_lower(k->n, k->Hres, ldk, 1, 0, k->st));
    CVXB_CUDA(cudaStreamSynchronize(k->st));
    return 0;
}

// --------------------------------------------------------------------- factor
int cvxb_kkt_factor(cvxb_kkt *k, const cvxb_scaling *Wp, const double *H, int ldh,
                    const double *Df, int lddf, int use_resident_H, int space) {
    if (!k) { set_error("kkt is NULL"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    if (k->method == 1) {
        if (H || Df || k->cone.mnl) { set_error("kkt_qr: the QR route solves systems with a zero (1,1) block (no H, no Df)"); return CVXB_E_ARG; }
        k->factored = false;
        int r = kkt_qr_factor(k, Wp, space);
        k->factored = (r == 0);
        return r;
    }
    const ConeLayout &c = k->cone;
    const int n = k->n;
    cudaStream_t st = k->st;
    k->factored = false;
    const long long ldk = kkt_ldk(k);
    CVXB_CUDA(cudaEventRecord(k->e0, st));
    CVXB_TRY(k->W.upload(c, Wp, space, st));
    const double *Hptr = nullptr;
    long long ldH = ldk;
    if (H) {
        if (ldh < (n > 1 ? n : 1)) { set_error("factor: ldh < n"); return CVXB_E_ARG; }
        if (space == CVXB_DEVICE) { Hptr = H; ldH = ldh; }
        else {
            if (!k->Hbuf) CVXB_CUDA(cudaMalloc(&k->Hbuf, (size_t)ldk * (n > 0 ? n : 1) * sizeof(double)));
            CVXB_TRY(upload_matrix(k->Hbuf, ldk, H, ldh, n, n, CVXB_HOST, st));
            Hptr = k->Hbuf;
        }
    } else if (use_resident_H && k->Hres) {
        Hptr = k->Hres;
    }
    // ---- Gs rows that cannot be folded into the SYRK operand load: [Df | q | s] ----
    if (c.mnl > 0) {
        if (!Df) { set_error("factor: Df is required when mnl > 0"); return CVXB_E_ARG; }
        const double *Dfd = Df; long long ldd = lddf;
        if (space != CVXB_DEVICE) {
            CVXB_TRY(upload_matrix(k->Dfbuf, c.mnl, Df, lddf, c.mnl, n, CVXB_HOST, st));
            Dfd = k->Dfbuf; ldd = c.mnl;
        }
        CVXB_TRY(scale_rows(Dfd, ldd, k->Gs, k->ldgs, c.mnl, n, k->W.dnli, st));
    }
    if (c.nq > 0)
        CVXB_TRY(scale_q(c, k->W, k->G + c.mnl + c.ml, k->ldg, k->Gs + c.mnl, k->ldgs, n, true, st));
    if (c.ns > 0) {
        // W^{-T} on an 's' block: rti' * mat(x) * rti  (trans 'T', inverse 'I'), then pack2
        CVXB_TRY(scale_s(c, k->W, k->G + c.mnl + c.ml + c.sumq, k->ldg, k->Gunp, c.sums2, n, 'T',
                         'I', k->swork, k->swork_doubles, st));
        CVXB_TRY(pack_s(c, k->Gunp, c.sums2, k->Gs + c.mnl + c.sumq, k->ldgs, n, false, st));
    }
    CVXB_CUDA(cudaEventRecord(k->e1, st));
    // ---- K = H + G_l' diag(di^2) G_l + Gs' Gs (+ A'A)  (lower triangle), then Cholesky ----
    int info = 0;
    auto assemble_and_factor = [&](bool add_ata) -> int {
        bool have = false;
        bool i8 = k->i8_mode == 2 || (k->i8_mode == 1 && n >= 4096 && c.ml >= 8192);
        if (c.ml > 0 && n > 0 && i8) {
            // the slice workspace is ~1.125 x sizeof(G_l): when it does not fit, the DMMA kernel (no
            // workspace) computes the same K
            const size_t need = ozaki_workspace_bytes(n, c.ml, 9);
            if (need > k->oz_bytes) {
                if (k->oz_work) cudaFree(k->oz_work);
                k->oz_work = nullptr; k->oz_bytes = 0;
                cudaError_t ae = cudaMalloc(&k->oz_work, need);
                if (ae == cudaErrorMemoryAllocation) { cudaGetLastError(); tmp_cache_release(); ae = cudaMalloc(&k->oz_work, need); }
                if (ae != cudaSuccess) {
                    cudaGetLastError();
                    k->oz_work = nullptr;
                    i8 = false;
                } else {
                    k->oz_bytes = need;
                }
            }
        }
        k->syrk_path = 0;
        if (c.ml > 0 && n > 0 && i8) {
            // G_l' diag(di)^2 G_l + H from nine int8 slices per entry (exact products, fp64-level result)
            ozaki_time_mma(k->m0, k->m1);
            CVXB_TRY(ozaki_syrk(n, c.ml, k->G + c.mnl, k->ldg, k->W.di, Hptr, ldH, 1.0, k->Kmat, ldk, 9, 0,
                                k->oz_work, nullptr, st));
            have = true;
            k->syrk_path = 2;
        } else if (c.ml > 0 && n > 0) {
            GemmDesc g;
            g.M = n; g.N = n; g.K = c.ml;
            g.X = k->G + c.mnl; g.ldx = (int)k->ldg; g.x_kmajor = true;
            g.Y = g.X; g.ldy = g.ldx; g.y_kmajor = true;
            g.w = k->W.di2;
            g.D = Hptr; g.ldd = (int)ldH; g.beta = 1.0;
            g.C = k->Kmat; g.ldc = (int)ldk;
            g.lower_only = true; g.splitk_ws = k->cw.splitk_ws;
            CVXB_TRY(dmma_gemm(g, st));
            have = true;
            k->syrk_path = 1;
        }
        if (k->nrest > 0 && n > 0) {
            GemmDesc g;
            g.M = n; g.N = n; g.K = k->nrest;
            g.X = k->Gs; g.ldx = (int)k->ldgs; g.x_kmajor = true;
            g.Y = g.X; g.ldy = g.ldx; g.y_kmajor = true;
            g.D = have ? k->Kmat : Hptr; g.ldd = have ? (int)ldk : (int)ldH; g.beta = 1.0;
            g.C = k->Kmat; g.ldc = (int)ldk;
            g.lower_only = true; g.splitk_ws = k->cw.splitk_ws;
            CVXB_TRY(dmma_gemm(g, st));
            have = true;
        }
        if (add_ata && k->p > 0 && n > 0) {
            GemmDesc g;                                   // S += A'A   (misc.py:1440)
            g.M = n; g.N = n; g.K = k->p;
            g.X = k->Aeq; g.ldx = (int)k->lda_eq; g.x_kmajor = true;
            g.Y = g.X; g.ldy = g.ldx; g.y_kmajor = true;
            g.D = have ? k->Kmat : Hptr; g.ldd = have ? (int)ldk : (int)ldH; g.beta = 1.0;
            g.C = k->Kmat; g.ldc = (int)ldk;
            g.lower_only = true; g.splitk_ws = k->cw.splitk_ws;
            CVXB_TRY(dmma_gemm(g, st));
            have = true;
        }
        if (!have && n > 0) {
            if (!Hptr) { set_error("factor: no cone rows and no H: KKT matrix is singular"); return 1; }
            CVXB_TRY(upload_matrix(k->Kmat, ldk, Hptr, ldH, n, n, CVXB_DEVICE, st));
        }
        CVXB_CUDA(cudaEventRecord(k->e2, st));
        if (k->method == 2 && k->p > 0) {
            // kkt_ldl2: Kmat now holds S = H + GG' W^-1 W^-T GG (lower); the 2x2 system [S A'; A 0] is factored
            // with Bunch-Kaufman pivoting (lapack.sytrf, misc.py:1172).  p == 0 is a plain Cholesky there too (:1173).
            CVXB_TRY(kkt_ldl_factor(k));
            CVXB_CUDA(cudaMemcpyAsync(&info, k->cw.d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
            CVXB_CUDA(cudaStreamSynchronize(st));
            return 0;
        }
        CVXB_TRY(potrf_lower(n, k->Kmat, (int)ldk, k->inv, k->cw, st));
        CVXB_CUDA(cudaMemcpyAsync(&info, k->cw.d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
        CVXB_CUDA(cudaStreamSynchronize(st));
        return 0;
    };
    CVXB_TRY(assemble_and_factor(k->method == 2 ? false : k->singular));
    if (info > 0 && k->p > 0 && k->first_factor && !k->singular && k->method != 2) {
        // S is singular on the first call: switch to S + A'A for the rest of the solve
        k->singular = true;
        info = 0;
        CVXB_TRY(assemble_and_factor(true));
    }
    k->first_factor = false;
    if (info == 0 && k->p > 0 && k->method != 2) {
        // Asct := L^{-1} A'  (blocked forward substitution with the diagonal-block inverses),
        // Kp := Asct' Asct,  Kp = Lp Lp'                               (misc.py:1464-1472)
        const int p = k->p;
        CVXB_TRY(transpose_copy(k->Aeq, k->lda_eq, k->Asct, k->ldas, p, n, st));
        CVXB_TRY(trsm_lower_left(n, k->Kmat, ldk, k->inv, k->Asct, k->ldas, p, st));
        {
            GemmDesc g;
            g.M = p; g.N = p; g.K = n;
            g.X = k->Asct; g.ldx = (int)k->ldas; g.x_kmajor = true;
            g.Y = k->Asct; g.ldy = (int)k->ldas; g.y_kmajor = true;
            g.C = k->Kp; g.ldc = (int)k->ldkp; g.lower_only = true;
            CVXB_TRY(dmma_gemm(g, st));
        }
        CVXB_TRY(potrf_lower(p, k->Kp, (int)k->ldkp, k->invp, k->cw, st));
        CVXB_CUDA(cudaMemcpyAsync(&info, k->cw.d_info, sizeof(int), cudaMemcpyDeviceToHost, st));
        CVXB_CUDA(cudaStreamSynchronize(st));
    }
    CVXB_CUDA(cudaEventRecord(k->e3, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    float t;
    cudaEventElapsedTime(&t, k->e0, k->e3); k->factor_ms = t;
    cudaEventElapsedTime(&t, k->e0, k->e1); k->br[0] = t;
    cudaEventElapsedTime(&t, k->e1, k->e2); k->br[1] = t;
    cudaEventElapsedTime(&t, k->e2, k->e3); k->br[2] = t;
    k->mma_ms = 0.0;
    if (k->syrk_path == 2 && k->method == 0 && cudaEventElapsedTime(&t, k->m0, k->m1) == cudaSuccess) k->mma_ms = t;
    cudaGetLastError();
    if (info > 0) {
        set_error("factor: leading minor of order %d is not positive definite", info);
        return info;
    }
    k->factored = true;
    return 0;
}

// --------------------------------------------------------------------- solve
int cvxb_kkt_solve(cvxb_kkt *k, double *x, double *y, double *z, int space) {
    if (!k) { set_error("kkt is NULL"); return CVXB_E_ARG; }
    if (!k->factored) { set_error("solve called before a successful factor"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    if (k->method == 1) return kkt_qr_solve(k, x, y, z, space);
    const ConeLayout &c = k->cone;
    const int n = k->n;
    cudaStream_t st = k->st;
    const long long ldk = kkt_ldk(k);
    const int nlq = c.mnl + c.ml + c.sumq;     // rows that are identical packed / unpacked
    CVXB_CUDA(cudaEventRecord(k->e0, st));
    double *xd = x, *zd = z, *ydv = y;
    if (k->p > 0 && !y) { set_error("solve: y is required when p > 0"); return CVXB_E_ARG; }
    if (space != CVXB_DEVICE) {
        CVXB_TRY(xfer_vec(k->xv, x, n, CVXB_HOST, true, st));
        CVXB_TRY(xfer_vec(k->zin, z, c.cdim, CVXB_HOST, true, st));
        xd = k->xv; zd = k->zin;
        if (k->p > 0) { CVXB_TRY(xfer_vec(k->yd, y, k->p, CVXB_HOST, true, st)); ydv = k->yd; }
    }
    CVXB_TRY(kkt_pack_bz(k, zd));
    // x := x + Gs' bzp                                            (misc.py:1311)
    if (c.ml > 0)
        CVXB_TRY(gemv_t(c.ml, n, k->G + c.mnl, k->ldg, k->W.di, k->bzp + c.mnl, 1.0, 1.0, xd, st));
    if (c.mnl > 0) CVXB_TRY(gemv_t(c.mnl, n, k->Gs, k->ldgs, nullptr, k->bzp, 1.0, 1.0, xd, st));
    if (k->nrest - c.mnl > 0)
        CVXB_TRY(gemv_t(k->nrest - c.mnl, n, k->Gs + c.mnl, k->ldgs, nullptr,
                        k->bzp + c.mnl + c.ml, 1.0, 1.0, xd, st));
    if (k->method == 2 && k->p > 0) {
        // [x; y] := (L D L')^{-1} [x; y]                          (lapack.sytrs, misc.py:1196)
        CVXB_TRY(kkt_ldl_solve(k, xd, ydv));
    } else if (k->p == 0) {
        // x := K^{-1} x                                           (misc.py:1327)
        CVXB_TRY(potrs_lower(n, k->Kmat, (int)ldk, k->inv, xd, k->cw, st));
    } else {
        // kkt_chol2-style elimination of the equality constraints  (misc.py:1526-1558)
        const int p = k->p;
        if (k->singular)      // x += A' by
            CVXB_TRY(gemv_t(p, n, k->Aeq, k->lda_eq, nullptr, ydv, 1.0, 1.0, xd, st));
        CVXB_TRY(trsv_lower(n, k->Kmat, (int)ldk, k->inv, xd, false, k->cw, st));          // x := L^{-1} x
        CVXB_TRY(gemv_t(n, p, k->Asct, k->ldas, nullptr, xd, 1.0, -1.0, ydv, st));         // y := Asct' x - y
        CVXB_TRY(potrs_lower(p, k->Kp, (int)k->ldkp, k->invp, ydv, k->cw, st));            // y := Kp^{-1} y
        CVXB_TRY(gemv_n(n, p, k->Asct, k->ldas, nullptr, ydv, -1.0, 1.0, xd, k->gemv_ws, st));   // x -= Asct y
        CVXB_TRY(trsv_lower(n, k->Kmat, (int)ldk, k->inv, xd, true, k->cw, st));           // x := L^{-T} x
    }
    // bzp := Gs x - bzp                                           (misc.py:1344)
    if (c.ml > 0)
        CVXB_TRY(gemv_n(c.ml, n, k->G + c.mnl, k->ldg, k->W.di, xd, 1.0, -1.0, k->bzp + c.mnl,
                        k->gemv_ws, st));
    if (c.mnl > 0)
        CVXB_TRY(gemv_n(c.mnl, n, k->Gs, k->ldgs, nullptr, xd, 1.0, -1.0, k->bzp, k->gemv_ws, st));
    if (k->nrest - c.mnl > 0)
        CVXB_TRY(gemv_n(k->nrest - c.mnl, n, k->Gs + c.mnl, k->ldgs, nullptr, xd, 1.0, -1.0,
                        k->bzp + c.mnl + c.ml, k->gemv_ws, st));
    CVXB_TRY(kkt_unpack_z(k, zd));
    if (space != CVXB_DEVICE) {
        CVXB_TRY(xfer_vec(x, k->xv, n, CVXB_HOST, false, st));
        CVXB_TRY(xfer_vec(z, k->zin, c.cdim, CVXB_HOST, false, st));
        if (k->p > 0) CVXB_TRY(xfer_vec(y, k->yd, k->p, CVXB_HOST, false, st));
    }
    CVXB_CUDA(cudaEventRecord(k->e1, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    float t;
    cudaEventElapsedTime(&t, k->e0, k->e1);
    k->solve_ms = t;
    return 0;
}

int cvxb_kkt_get_L(cvxb_kkt *k, double *L_host, int ldl) {
    if (!k || !L_host || ldl < k->n) { set_error("get_L: bad arguments"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    CVXB_CUDA(cudaMemcpy2D(L_host, (size_t)ldl * sizeof(double), k->Kmat, kkt_ldk(k) * sizeof(double),
                           (size_t)k->n * sizeof(double), k->n, cudaMemcpyDeviceToHost));
    return 0;
}

int cvxb_kkt_last_ms(cvxb_kkt *k, double *factor_ms, double *solve_ms) {
    if (!k) return CVXB_E_ARG;
    if (factor_ms) *factor_ms = k->factor_ms;
    if (solve_ms) *solve_ms = k->solve_ms;
    return 0;
}
int cvxb_kkt_timer_start(cvxb_kkt *k) {
    if (!k) return CVXB_E_ARG;
    CVXB_CUDA(cudaSetDevice(k->device));
    CVXB_CUDA(cudaStreamSynchronize(k->st));
    CVXB_CUDA(cudaEventRecord(k->t0, k->st));
    return 0;
}
int cvxb_kkt_timer_stop(cvxb_kkt *k, double *ms) {
    if (!k || !ms) return CVXB_E_ARG;
    CVXB_CUDA(cudaSetDevice(k->device));
    CVXB_CUDA(cudaEventRecord(k->t1, k->st));
    CVXB_CUDA(cudaEventSynchronize(k->t1));
    float t = 0;
    CVXB_CUDA(cudaEventElapsedTime(&t, k->t0, k->t1));
    *ms = t;
    return 0;
}
/* debug: copy the CVXB_TRACE timeline of the last potrf (8 values per block step) */
int cvxb_kkt_trace(cvxb_kkt *k, unsigned long long *out, int nsteps) {
    if (!k || !out || !k->cw.trace) return CVXB_E_ARG;
    CVXB_CUDA(cudaMemcpy(out, k->cw.trace, (size_t)nsteps * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}
int cvxb_kkt_syrk_path(cvxb_kkt *k) { return k ? k->syrk_path : CVXB_E_ARG; }
int cvxb_kkt_qr_passes(cvxb_kkt *k) { return (k && k->method == 1) ? kkt_qr_passes(k) : CVXB_E_ARG; }
int cvxb_kkt_last_breakdown(cvxb_kkt *k, double *ms3) {
    if (!k || !ms3) return CVXB_E_ARG;
    ms3[0] = k->br[1]; ms3[1] = k->br[2]; ms3[2] = k->br[0];
    return 0;
}

int cvxb_kkt_syrk_mma_ms(cvxb_kkt *k, double *ms) {
    if (!k || !ms) return CVXB_E_ARG;
    *ms = k->mma_ms;
    return 0;
}

int cvxb_kkt_gemv_G(cvxb_kkt *k, const double *x, double *y, double alpha, double beta, int trans,
                    int space) {
    if (!k || !x || !y) { set_error("gemv_G: bad arguments"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    const ConeLayout &c = k->cone;
    const int n = k->n, m = c.cdim - c.mnl;
    cudaStream_t st = k->st;
    const double *Gp = k->G + c.mnl;
    const bool tr = (trans == 'T' || trans == 't');
    const int nx = tr ? m : n, ny = tr ? n : m;
    const double *xd = x; double *yd = y;
    if (space != CVXB_DEVICE) {
        // zin/yv are cdim long, xv is n long: pick by role
        double *xb = tr ? k->zin : k->xv, *yb = tr ? k->xv : k->yv;
        CVXB_TRY(xfer_vec(xb, x, nx, CVXB_HOST, true, st));
        if (beta != 0.0) CVXB_TRY(xfer_vec(yb, y, ny, CVXB_HOST, true, st));
        xd = xb; yd = yb;
    }
    if (tr) CVXB_TRY(gemv_t(m, n, Gp, k->ldg, nullptr, xd, alpha, beta, yd, st));
    else    CVXB_TRY(gemv_n(m, n, Gp, k->ldg, nullptr, xd, alpha, beta, yd, k->gemv_ws, st));
    if (space != CVXB_DEVICE) CVXB_TRY(xfer_vec(y, yd, ny, CVXB_HOST, false, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int cvxb_kkt_gemv_A(cvxb_kkt *k, const double *x, double *y, double alpha, double beta, int trans,
                    int space) {
    if (!k || !x || !y) { set_error("gemv_A: bad arguments"); return CVXB_E_ARG; }
    if (k->p <= 0) { set_error("gemv_A: the factory was created without equality constraints"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    const int n = k->n, p = k->p;
    cudaStream_t st = k->st;
    const bool tr = (trans == 'T' || trans == 't');
    const int nx = tr ? p : n, ny = tr ? n : p;
    const double *xd = x; double *yd = y;
    if (space != CVXB_DEVICE) {
        // xv (n) / yd (p) by role; yv is max(cdim, n) long and serves as the second n- or p-vector
        double *xb = tr ? k->yd : k->xv, *yb = k->yv;
        if (!tr && p > n) { set_error("gemv_A: p > n"); return CVXB_E_ARG; }
        CVXB_TRY(xfer_vec(xb, x, nx, CVXB_HOST, true, st));
        if (beta != 0.0) CVXB_TRY(xfer_vec(yb, y, ny, CVXB_HOST, true, st));
        xd = xb; yd = yb;
    }
    if (tr) CVXB_TRY(gemv_t(p, n, k->Aeq, k->lda_eq, nullptr, xd, alpha, beta, yd, st));
    else    CVXB_TRY(gemv_n(p, n, k->Aeq, k->lda_eq, nullptr, xd, alpha, beta, yd, k->gemv_ws, st));
    if (space != CVXB_DEVICE) CVXB_TRY(xfer_vec(y, yd, ny, CVXB_HOST, false, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

int cvxb_kkt_symv_H(cvxb_kkt *k, const double *x, double *y, double alpha, double beta, int space) {
    if (!k || !x || !y) { set_error("symv_H: bad arguments"); return CVXB_E_ARG; }
    if (!k->Hres) { set_error("symv_H: no resident H (call cvxb_kkt_set_H)"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(k->device));
    const int n = k->n;
    cudaStream_t st = k->st;
    const double *xd = x; double *yd = y;
    if (space != CVXB_DEVICE) {
        CVXB_TRY(xfer_vec(k->xv, x, n, CVXB_HOST, true, st));
        if (beta != 0.0) CVXB_TRY(xfer_vec(k->yv, y, n, CVXB_HOST, true, st));
        xd = k->xv; yd = k->yv;
    }
    CVXB_TRY(gemv_t(n, n, k->Hres, kkt_ldk(k), nullptr, xd, alpha, beta, yd, st));
    if (space != CVXB_DEVICE) CVXB_TRY(xfer_vec(y, yd, n, CVXB_HOST, false, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    return 0;
}

}  // extern "C"
