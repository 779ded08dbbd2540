// Device-resident primal-dual interior-point method for a BATCH of independent dense QPs
//
//      minimize  1/2 x'P x + q'x    subject to  G x + s = h,  s >= 0,  A x = b      ('l' cone, p >= 0 rows of A)
//
// run in lock-step, one problem per CTA-group, with per-problem convergence masks
// (BASELINE config 4; the reference has no batch API — its counterpart is a Python loop over
// solvers.qp).  The algorithm is a restatement of coneprog.coneqp for dims = {'l': m}
// (reference src/python/coneprog.py:1998-2547): same starting point (:2055-2106), residuals
// and stopping rule (:2169-2234), Nesterov-Todd scaling d = sqrt(s/z) (misc.py:284-287),
// Mehrotra predictor/corrector with STEP 0.99 / EXPON 3 (:2357-2456) and scaling update
// (misc.py:450-464).  Every KKT solve is the same path as cvxb_kkt_*: fused-scaling SYRK,
// Cholesky, GEMV/TRSV — here batched over the problems through blockIdx.z / blockIdx.y.
// Nothing leaves the device between iterations except one int ("how many are done").
//
// Equality constraints (p > 0) are eliminated as the reference's default KKT solver for this case does,
// misc.kkt_chol2 (misc.py:1352-1567): S = P + G' D^-2 G = L L', Asct = L^{-1} A', Kp = Asct' Asct = Lp Lp'.
// A problem whose S is singular at the starting point (W = I) factors S + A'A from then on (misc.py:1421-1461);
// per problem, through a 0/1 weight vector of length p (`wsing`) applied inside the batched GEMM / GEMV.
//
// Second-order cones: the inequality rows may be dims = {'l': ml, 'q': [q_1 .. q_K]} (the same for every problem), and
// the algorithm is then coneqp with that dims and its default options (:1805-1809, :1862-1865): one step of iterative
// refinement per Newton solve (f4, :2330-2347; any count through options['refinement'], for 'l'-only batches too) and
// the same kkt_chol2 elimination, with the cones' rows scaled explicitly (Gs_q = W^{-T} G_q) and added to S by a second
// batched GEMM.  The cone kernels walk a problem's cones with one thread, a warp or the CTA per cone (GThread / GWarp /
// GBlock below), chosen at create from the cone sizes.
#include "kkt_internal.cuh"
#include <algorithm>
#include <cstdlib>

using namespace cvxb;

namespace {

struct Scal {                       // per-problem scalars, device resident
    double resx0, resz0, gap, mu, sigma, eta, step, dsdz;
    double xPxq, xq, resx, resz, zrz, pcost, dcost, relgap, pres, dres;
    double resy0, resy, yry;                 // equality constraints: max(1, ||b||), ||A x - b||, y'(A x - b)
    int relgap_valid, done, iters, status;   // status: 0 running, 1 optimal, 2 maxiters, 3 singular
    int singular, pad_;                      // singular: S + A'A is factored (kkt_chol2's F['singular'])
};

__device__ __forceinline__ double block_sum(double v, double *sh) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
    if (warp == 0) t = warp_sum(t);
    if (threadIdx.x == 0) sh[0] = t;
    __syncthreads();
    return sh[0];
}
__device__ __forceinline__ double block_min(double v, double *sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : INFINITY;
    if (warp == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t = fmin(t, __shfl_xor_sync(0xffffffffu, t, o));
    }
    if (threadIdx.x == 0) sh[0] = t;
    __syncthreads();
    return sh[0];
}
__device__ __forceinline__ double block_max(double v, double *sh) { return -block_min(-v, sh); }

// ---- 'q' cones: the threads that work on one cone ("group") ----
// Every problem has the same cones; a CTA (one problem) walks them with groups of 1 thread (tiny cones), a warp
// (many cones) or the whole CTA (a few large cones).  Group g takes cones g, g + ngroups, ...; element i of a cone
// belongs to the group's thread i mod size, and element 0 to rank 0.  sum() reduces over the group and returns the
// total to every member; it orders the members' earlier global writes before their later reads.
struct GThread {
    __device__ int rank() const { return 0; }
    __device__ int size() const { return 1; }
    __device__ int gid() const { return threadIdx.x; }
    __device__ int ngroups() const { return blockDim.x; }
    __device__ double sum(double v, double *) const { return v; }
    __device__ void sync() const {}
};
struct GWarp {
    __device__ int rank() const { return threadIdx.x & 31; }
    __device__ int size() const { return 32; }
    __device__ int gid() const { return threadIdx.x >> 5; }
    __device__ int ngroups() const { return blockDim.x >> 5; }
    __device__ double sum(double v, double *) const { __syncwarp(); v = warp_sum(v); __syncwarp(); return v; }
    __device__ void sync() const { __syncwarp(); }
};
struct GBlock {
    __device__ int rank() const { return threadIdx.x; }
    __device__ int size() const { return blockDim.x; }
    __device__ int gid() const { return 0; }
    __device__ int ngroups() const { return 1; }
    __device__ double sum(double v, double *sh) const { return block_sum(v, sh); }
    __device__ void sync() const { __syncthreads(); }
};

// Per-cone formulas of the reference's cone algebra (misc_solvers.c / misc.py, cited at each helper), in the same
// arithmetic as the single-problem kernels of cone_vec.cu, nt_scaling.cu and cone.cu.  x, y, ... point at the cone's
// first element; mq is its size.  Every helper ends with the group synchronised.

// max_step of one cone: ||x1|| - x0  (misc_solvers.c:1083-1093)
template <class Gp>
__device__ double q_max_step(const Gp &g, const double *x, int mq, double *sh) {
    double n2 = 0;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) n2 += x[i] * x[i];
    n2 = g.sum(n2, sh);
    return sqrt(n2) - x[0];
}
// x := y o\ x  (sinv, misc_solvers.c:813-850)
template <class Gp>
__device__ void q_sinv(const Gp &g, double *x, const double *y, int mq, double *sh) {
    double n2 = 0, d = 0;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) { n2 += y[i] * y[i]; d += x[i] * y[i]; }
    const double y0 = y[0], cx = x[0];
    n2 = g.sum(n2, sh); d = g.sum(d, sh);
    const double nrm = sqrt(n2);
    const double a = (y0 + nrm) * (y0 - nrm);
    const double al1 = a / y0, al2 = d / y0 - cx, ia = 1.0 / a;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) x[i] = (x[i] * al1 + al2 * y[i]) * ia;
    if (g.rank() == 0) x[0] = (cx * y0 - d) * ia;
    g.sync();
}
// x := y o x  (sprod, misc_solvers.c:680-700; the same with diag = 'D')
template <class Gp>
__device__ void q_sprod(const Gp &g, double *x, const double *y, int mq, double *sh) {
    double d = 0;
    for (int i = g.rank(); i < mq; i += g.size()) d += y[i] * x[i];
    const double y0 = y[0], x0 = x[0];
    d = g.sum(d, sh);
    for (int i = 1 + g.rank(); i < mq; i += g.size()) x[i] = y0 * x[i] + x0 * y[i];
    if (g.rank() == 0) x[0] = d;
    g.sync();
}
// x := W x = beta (2 v v' - J) x,  or  x := W^{-1} x = (1/beta) (2 J v v' J - J) x  (scale, misc_solvers.c:156-183)
template <class Gp>
__device__ void q_scale(const Gp &g, double *x, const double *v, double beta, int mq, bool inverse, double *sh) {
    double w = 0;
    for (int i = g.rank(); i < mq; i += g.size()) {
        double xi = x[i];
        if (inverse && i == 0) xi = -xi;
        w += v[i] * xi;
    }
    w = g.sum(w, sh);
    const double tw = 2.0 * w, bb = inverse ? 1.0 / beta : beta;
    for (int i = g.rank(); i < mq; i += g.size()) {
        double xi = x[i];
        if (!inverse && i == 0) xi = -xi;
        double yi = xi + v[i] * tw;
        if (inverse && i == 0) yi = -yi;
        x[i] = yi * bb;
    }
    g.sync();
}
// x := H(lambda^{1/2}) x or its inverse  (scale2, misc_solvers.c:296-335)
template <class Gp>
__device__ void q_scale2(const Gp &g, const double *lm, double *x, int mq, bool inverse, double *sh) {
    double n2 = 0, dot = 0;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) { n2 += lm[i] * lm[i]; dot += lm[i] * x[i]; }
    const double l0 = lm[0], x0 = x[0];
    n2 = g.sum(n2, sh); dot = g.sum(dot, sh);
    const double nrm = sqrt(n2);
    const double a = sqrt(l0 + nrm) * sqrt(l0 - nrm);
    const double lx = inverse ? (l0 * x0 + dot) / a : (l0 * x0 - dot) / a;
    double c = (x0 + lx) / (l0 / a + 1.0) / a;
    if (!inverse) c = -c;
    const double sc = inverse ? a : 1.0 / a;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) x[i] = (x[i] + c * lm[i]) * sc;
    if (g.rank() == 0) x[0] = lx * sc;
    g.sync();
}
// out := lambda o lambda  (ssqr, misc.py:957-962)
template <class Gp>
__device__ void q_ssqr(const Gp &g, double *out, const double *lm, int mq, double *sh) {
    double n2 = 0;
    for (int i = g.rank(); i < mq; i += g.size()) n2 += lm[i] * lm[i];
    n2 = g.sum(n2, sh);
    const double l0 = lm[0];
    for (int i = 1 + g.rank(); i < mq; i += g.size()) out[i] = 2.0 * l0 * lm[i];
    if (g.rank() == 0) out[0] = n2;
    g.sync();
}
// sqrt(x' J x) as misc.jnrm2 evaluates it (misc.py:848-856)
template <class Gp>
__device__ double q_jnrm2(const Gp &g, const double *x, int mq, double *sh) {
    double t = 0;
    for (int i = 1 + g.rank(); i < mq; i += g.size()) t += x[i] * x[i];
    const double x0 = x[0];
    const double a = sqrt(g.sum(t, sh));
    return sqrt(x0 - a) * sqrt(x0 + a);
}
// Nesterov-Todd scaling of one cone from s, z: v, beta, lambda  (compute_scaling, misc.py:311-354)
template <class Gp>
__device__ void q_compute_scaling(const Gp &g, const double *sk, const double *zk, double *v, double *beta,
                                  double *lk, int mq, double *sh) {
    const double aa = q_jnrm2(g, sk, mq, sh), bb = q_jnrm2(g, zk, mq, sh);
    double t = 0;
    for (int i = g.rank(); i < mq; i += g.size()) t += sk[i] * zk[i];
    const double dot = g.sum(t, sh);
    const double cc = sqrt((dot / aa / bb + 1.0) / 2.0);
    const double s0 = sk[0], z0 = zk[0];
    const double v0 = ((s0 / aa) + (z0 / bb)) / 2.0 / cc + 1.0;
    const double sc = 1.0 / sqrt(2.0 * v0);
    const double dd = 2.0 * cc + s0 / aa + z0 / bb;
    const double c1 = (cc + z0 / bb) / dd / aa, c2 = (cc + s0 / aa) / dd / bb, sab = sqrt(aa * bb);
    for (int i = g.rank(); i < mq; i += g.size()) {
        if (i == 0) {
            v[0] = v0 * sc;
            lk[0] = cc * sab;
        } else {
            v[i] = ((sk[i] / aa - zk[i] / bb) / 2.0 / cc) * sc;
            lk[i] = (c1 * sk[i] + c2 * zk[i]) * sab;
        }
    }
    if (g.rank() == 0) *beta = sqrt(aa / bb);
    g.sync();
}
// scaling update of one cone; sk, zk hold the new iterates in the current scaling and are normalised in place
// (update_scaling, misc.py:504-573)
template <class Gp>
__device__ void q_update_scaling(const Gp &g, double *sk, double *zk, double *v, double *beta, double *lk, int mq,
                                 double *sh) {
    const double aa = q_jnrm2(g, sk, mq, sh);
    for (int i = g.rank(); i < mq; i += g.size()) sk[i] *= 1.0 / aa;
    g.sync();
    const double bb = q_jnrm2(g, zk, mq, sh);
    for (int i = g.rank(); i < mq; i += g.size()) zk[i] *= 1.0 / bb;
    g.sync();
    double t1 = 0, t2 = 0, t3 = 0;
    for (int i = g.rank(); i < mq; i += g.size()) {
        t1 += sk[i] * zk[i];
        t2 += v[i] * sk[i];
        t3 += (i == 0 ? v[i] * zk[i] : -v[i] * zk[i]);     // jdot: v' J z
    }
    const double s0 = sk[0], z0 = zk[0], vk0 = v[0];
    const double dot = g.sum(t1, sh), vs = g.sum(t2, sh), vz = g.sum(t3, sh);
    const double cc = sqrt((1.0 + dot) / 2.0);
    const double vq = (vs + vz) / 2.0 / cc, vu = vs - vz;
    const double wk0 = 2.0 * vk0 * vq - (s0 + z0) / 2.0 / cc;
    const double dd = (vk0 * vu - s0 / 2.0 + z0 / 2.0) / (wk0 + 1.0);
    const double sab = sqrt(aa * bb);
    const double vn0 = 2.0 * vq * vk0 - s0 / 2.0 / cc - 0.5 / cc * z0 + 1.0;
    const double sc = 1.0 / sqrt(2.0 * vn0);
    for (int i = g.rank(); i < mq; i += g.size()) {
        const double vi = v[i], si = sk[i], zi = zk[i];
        if (i == 0) {
            lk[0] = cc * sab;
            v[0] = vn0 * sc;
        } else {
            lk[i] = (vi * (2.0 * (-dd * vq + 0.5 * vu)) + 0.5 * (1.0 - dd / cc) * si + 0.5 * (1.0 + dd / cc) * zi) * sab;
            v[i] = (2.0 * vq * vi + 0.5 / cc * si - 0.5 / cc * zi) * sc;
        }
    }
    if (g.rank() == 0) *beta *= sqrt(aa / bb);
    g.sync();
}

// the cone table: sizes and offsets (within the 'q' rows) of the K cones, the same for every problem
struct QCones {
    int ml, nq, sumq;               // 'l' rows, number of 'q' cones, their total size
    const int *dim, *off;           // device arrays of length nq
    const double *e;                // sumq: 1 at the first row of every cone, else 0 (the identity of the cone)
    double *vb;                     // per problem (stride sumq + nq): v of every cone, then beta of every cone
};

struct Ptrs {
    int n, m, neq;                  // neq: rows of A (p)
    const double *q, *h, *beq;
    double *x, *s, *z, *rx, *rz, *dx, *ds, *dz, *lmbda, *lmbdasq, *d, *di, *di2, *ws3, *bzp;
    double *y, *ry, *dy, *wsing;    // p-vectors (wsing: 1 where S + A'A is factored, else 0)
    Scal *sc;
    QCones c;
    // iterative refinement (allocated by the first solve that asks for it): the right-hand side of the Newton
    // system (wx wy wz ws), the correction's right-hand side / solution (x2 y2 z2 s2), W^{-1} uz (t3)
    double *wx, *wy, *wz, *ws, *x2, *y2, *z2, *s2, *t3;
};
// cone k of problem b:  rows  om + ml + off[k]  of an m-vector;  v at vb + b (sumq + nq) + off[k]
#define Q_CONE(k)                                                          \
    const int mq = p.c.dim[k];                                             \
    const long long oq = om + p.c.ml + p.c.off[k];                         \
    double *vq_ = p.c.vb + (long long)b * (p.c.sumq + p.c.nq) + p.c.off[k]; \
    double *betaq_ = p.c.vb + (long long)b * (p.c.sumq + p.c.nq) + p.c.sumq + k;
#define Q_LOOP(g) for (int k = (g).gid(); k < p.c.nq; k += (g).ngroups())
#define PB_SETUP                                                  \
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x; \
    const long long on = (long long)b * p.n, om = (long long)b * p.m; \
    __shared__ double sh[32];                                     \
    Scal &S = p.sc[b];

// starting point, part 1: rhs of [P G'; G -I][x; z] = [-q; h] with W = I   (coneprog.py:2076-2080)
__global__ void k_init_rhs(Ptrs p) {
    PB_SETUP
    double nq = 0, nh = 0;
    for (int i = tid; i < p.n; i += nt) { double v = p.q[on + i]; p.dx[on + i] = -v; nq += v * v; }
    for (int i = tid; i < p.m; i += nt) {
        double v = p.h[om + i];
        p.dz[om + i] = v;
        p.d[om + i] = 1.0; p.di[om + i] = 1.0; p.di2[om + i] = 1.0;
        nh += v * v;
    }
    nq = block_sum(nq, sh);
    nh = block_sum(nh, sh);
    double nb = 0;
    if (p.neq > 0) {                                    // dy = b
        const long long op = (long long)b * p.neq;
        for (int i = tid; i < p.neq; i += nt) { double v = p.beq[op + i]; p.dy[op + i] = v; nb += v * v; }
        nb = block_sum(nb, sh);
    }
    if (p.c.nq > 0) {                                   // W = I: v = e, beta = 1 (:2058-2060)
        double *vb = p.c.vb + (long long)b * (p.c.sumq + p.c.nq);
        for (int i = tid; i < p.c.sumq; i += nt) vb[i] = p.c.e[i];
        for (int k = tid; k < p.c.nq; k += nt) vb[p.c.sumq + k] = 1.0;
    }
    if (tid == 0) {
        S.resx0 = fmax(1.0, sqrt(nq));                  // :1998
        S.resy0 = fmax(1.0, sqrt(nb));                  // :1999
        S.resz0 = fmax(1.0, sqrt(nh));                  // :2000 (snrm2 == 2-norm for 'l')
        S.done = 0; S.iters = 0; S.status = 0; S.sigma = 0; S.eta = 0; S.step = 0;
    }
}
// bzp = di .* bz  (W^{-T} bz for the 'l' cone)
__global__ void k_scale_bz(Ptrs p, const double *bz) {
    PB_SETUP
    (void)sh; (void)S; (void)on;
    for (int i = tid; i < p.m; i += nt) p.bzp[om + i] = p.di[om + i] * bz[om + i];
}
// starting point, part 2: x = dx, z = dz (solution), s = -z, shifts (:2083-2106), gap (:2165)
template <class Gp>
__global__ void k_init_point(Ptrs p) {
    PB_SETUP
    const int ml = p.c.ml;
    double ns = 0, mins = INFINITY;
    for (int i = tid; i < p.n; i += nt) p.x[on + i] = p.dx[on + i];
    const long long op = (long long)b * p.neq;
    for (int i = tid; i < p.neq; i += nt) p.y[op + i] = p.dy[op + i];
    for (int i = tid; i < p.m; i += nt) {
        double zv = p.bzp[om + i];      // solve leaves W*uz in bzp
        p.z[om + i] = zv;
        p.s[om + i] = -zv;
        ns += zv * zv;                  // snrm2 == 2-norm for 'l' and 'q'
        if (i < ml) mins = fmin(mins, -zv);
    }
    ns = sqrt(block_sum(ns, sh));
    mins = block_min(mins, sh);
    double ts = -mins;                                   // max_step(s) = -min(s) for 'l'
    double minz = INFINITY;
    for (int i = tid; i < ml; i += nt) minz = fmin(minz, p.z[om + i]);
    minz = block_min(minz, sh);
    double tz = -minz;
    if (p.c.nq > 0) {                                    // and max over the cones of ||x1|| - x0
        const Gp g;
        double tsq = -INFINITY, tzq = -INFINITY;
        Q_LOOP(g) {
            Q_CONE(k) (void)vq_; (void)betaq_;
            tsq = fmax(tsq, q_max_step(g, p.s + oq, mq, sh));
            tzq = fmax(tzq, q_max_step(g, p.z + oq, mq, sh));
        }
        ts = fmax(ts, block_max(tsq, sh));
        tz = fmax(tz, block_max(tzq, sh));
    }
    const double as = (ts >= -1e-8 * fmax(ns, 1.0)) ? 1.0 + ts : 0.0;
    const double az = (tz >= -1e-8 * fmax(ns, 1.0)) ? 1.0 + tz : 0.0;   // nrmz == nrms here
    double gap = 0;
    for (int i = tid; i < p.m; i += nt) {
        const double e = i < ml ? 1.0 : p.c.e[i - ml];  // every 'l' row, the first row of every cone
        double sv = p.s[om + i] + as * e, zv = p.z[om + i] + az * e;
        p.s[om + i] = sv; p.z[om + i] = zv;
        gap += sv * zv;
    }
    gap = block_sum(gap, sh);
    if (tid == 0) S.gap = gap;
}
// rx = q  (then rx += P x by GEMV); ry = b (then ry := A x - ry)
__global__ void k_res_begin(Ptrs p) {
    PB_SETUP
    (void)sh; (void)S;
    for (int i = tid; i < p.n; i += nt) p.rx[on + i] = p.q[on + i];
    for (int i = tid; i < p.m; i += nt) p.rz[om + i] = p.s[om + i] - p.h[om + i];      // :2183-2184
    const long long op = (long long)b * p.neq;
    for (int i = tid; i < p.neq; i += nt) p.ry[op + i] = p.beq[op + i];                 // :2178
}
// f0 pieces once rx = P x + q   (:2172)
__global__ void k_res_dots(Ptrs p) {
    PB_SETUP
    double a = 0, c = 0;
    for (int i = tid; i < p.n; i += nt) { double xv = p.x[on + i]; a += xv * p.rx[on + i]; c += xv * p.q[on + i]; }
    a = block_sum(a, sh); c = block_sum(c, sh);
    if (tid == 0) { S.xPxq = a; S.xq = c; }
}
// statistics + stopping rule (:2175-2234)
__global__ void k_stats(Ptrs p, int iter, int maxiters, double abstol, double reltol, double feastol,
                        int *ndone, int *doneflags) {
    PB_SETUP
    double rx2 = 0, rz2 = 0, zrz = 0;
    for (int i = tid; i < p.n; i += nt) { double v = p.rx[on + i]; rx2 += v * v; }
    for (int i = tid; i < p.m; i += nt) { double v = p.rz[om + i]; rz2 += v * v; zrz += p.z[om + i] * v; }
    rx2 = block_sum(rx2, sh); rz2 = block_sum(rz2, sh); zrz = block_sum(zrz, sh);
    double ry2 = 0, yry = 0;
    if (p.neq > 0) {
        const long long op = (long long)b * p.neq;
        for (int i = tid; i < p.neq; i += nt) { double v = p.ry[op + i]; ry2 += v * v; yry += p.y[op + i] * v; }
        ry2 = block_sum(ry2, sh); yry = block_sum(yry, sh);
    }
    if (tid == 0) {
        if (!S.done) {
            const double f0 = 0.5 * (S.xPxq + S.xq);
            S.resx = sqrt(rx2); S.resz = sqrt(rz2); S.zrz = zrz;
            S.resy = sqrt(ry2); S.yry = yry;
            S.pcost = f0;
            S.dcost = (p.neq > 0 ? f0 + yry : f0) + zrz - S.gap;
            if (S.pcost < 0.0) { S.relgap = S.gap / -S.pcost; S.relgap_valid = 1; }
            else if (S.dcost > 0.0) { S.relgap = S.gap / S.dcost; S.relgap_valid = 1; }
            else { S.relgap = 0.0; S.relgap_valid = 0; }
            S.pres = p.neq > 0 ? fmax(S.resy / S.resy0, S.resz / S.resz0) : S.resz / S.resz0;
            S.dres = S.resx / S.resx0;
            const bool opt = S.pres <= feastol && S.dres <= feastol &&
                             (S.gap <= abstol || (S.relgap_valid && S.relgap <= reltol));
            if (opt || iter == maxiters) {
                S.done = 1; S.iters = iter; S.status = opt ? 1 : 2;
            }
        }
        if (S.done) atomicAdd(ndone, 1);
        doneflags[b] = S.done;
    }
}

// ---- compaction of finished problems ----
// The lock-step loop launches every batched kernel over the first `Bact` slots.  When problems finish, each finished
// slot below the new active count trades places with an active slot from the tail: everything a problem owns between
// iterations (P, G, A, its 17 + 5 vectors, v and beta of its cones, its scalars; K / inv / info / Asct / Kp / Gs_q and
// the refinement vectors are rebuilt every iteration) is swapped,
// so the active
// problems stay a contiguous prefix and finished ones keep their final iterates in the tail.  ~6.3 MB per swap at
// n=512, m=1024 (p = 0), at most one swap per problem per solve.
struct SwapArgs {
    double *P, *G, *vecs, *A, *veq, *vb; Scal *sc;
    long long sP, sG, sA;
    int n, me, neq, nvb, Btot;      // nvb: v and beta of the 'q' cones (sumq + nq, 0 without cones)
};
__global__ void k_swap_slots(SwapArgs a, const int *pairs) {
    const int i = pairs[2 * blockIdx.y], j = pairs[2 * blockIdx.y + 1];
    const long long eP = a.sP, eG = a.sG, eN = 4LL * a.n, eM = 13LL * a.me, eS = (long long)(sizeof(Scal) / sizeof(double));
    const long long eA = a.sA, eQ = 5LL * a.neq;          // both 0 without equality constraints
    const long long eV = a.nvb;
    const long long total = eP + eG + eN + eM + eS + eA + eQ + eV;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        double *x, *y;
        long long r = e;
        if (r < eP) { x = a.P + i * a.sP + r; y = a.P + j * a.sP + r; }
        else if ((r -= eP) < eG) { x = a.G + i * a.sG + r; y = a.G + j * a.sG + r; }
        else if ((r -= eG) < eN) {
            const long long arr = r / a.n, k = r % a.n;
            double *base = a.vecs + arr * (long long)a.Btot * a.n;
            x = base + (long long)i * a.n + k; y = base + (long long)j * a.n + k;
        } else if ((r -= eN) < eM) {
            const long long arr = r / a.me, k = r % a.me;
            double *base = a.vecs + 4LL * a.Btot * a.n + arr * (long long)a.Btot * a.me;
            x = base + (long long)i * a.me + k; y = base + (long long)j * a.me + k;
        } else if ((r -= eM) < eS) {
            x = reinterpret_cast<double *>(a.sc + i) + r; y = reinterpret_cast<double *>(a.sc + j) + r;
        } else if ((r -= eS) < eA) {
            x = a.A + i * a.sA + r; y = a.A + j * a.sA + r;
        } else if ((r -= eA) >= eQ) {
            r -= eQ;
            x = a.vb + (long long)i * a.nvb + r; y = a.vb + (long long)j * a.nvb + r;
        } else {
            const long long arr = r / a.neq, k = r % a.neq;
            double *base = a.veq + arr * (long long)a.Btot * a.neq;
            x = base + (long long)i * a.neq + k; y = base + (long long)j * a.neq + k;
        }
        const double t = *x; *x = *y; *y = t;
    }
}
// out[perm[slot], :] = in[slot, :]
__global__ void k_unpermute_rows(const double *in, double *out, const int *perm, int len) {
    const int slot = blockIdx.x;
    const double *src = in + (long long)slot * len;
    double *dst = out + (long long)perm[slot] * len;
    for (int k = threadIdx.x; k < len; k += blockDim.x) dst[k] = src[k];
}
static_assert(sizeof(Scal) % sizeof(double) == 0, "Scal is swapped as doubles");

// kkt_chol2's first factorisation (misc.py:1421-1447): a problem whose S did not factor at the starting point is
// flagged, and S + A'A is factored for it from then on.  info: one int per problem from the Cholesky of S.
__global__ void k_flag_singular(Ptrs p, const int *info, int *nsing) {
    const int b = blockIdx.x;
    if (info[b] <= 0) return;
    const long long op = (long long)b * p.neq;
    for (int k = threadIdx.x; k < p.neq; k += blockDim.x) p.wsing[op + k] = 1.0;
    if (threadIdx.x == 0) { p.sc[b].singular = 1; atomicAdd(nsing, 1); }
}
// a failed Cholesky of Kp counts as a failed factorisation of the problem (the reference raises either way)
__global__ void k_fold_info(const int *infop, int *info, int n, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B && info[b] <= 0 && infop[b] > 0) info[b] = n + infop[b];
}
// Asct := A'  (p x n, ld lda  ->  n x p, ld ldas), every problem of the batch (blockIdx.y)
__global__ void k_transpose_A(const double *A, long long lda, long long sA, double *At, long long ldas, long long sAt,
                              int n, int neq) {
    const long long b = blockIdx.y, tot = (long long)n * neq;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e % n, k = e / n;
        At[b * sAt + i + k * ldas] = A[b * sA + k + i * lda];
    }
}
// NT scaling at iteration 0 (misc.py:284-287, 'q': :311-354) and lambda^2 (:2244)
template <class Gp>
__global__ void k_scaling(Ptrs p, int first) {
    PB_SETUP
    (void)on;
    if (S.done) return;
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k)
            if (first) q_compute_scaling(g, p.s + oq, p.z + oq, vq_, betaq_, p.lmbda + oq, mq, sh);
            q_ssqr(g, p.lmbdasq + oq, p.lmbda + oq, mq, sh);
        }
    }
    for (int i = tid; i < p.c.ml; i += nt) {
        if (first) {
            const double sv = p.s[om + i], zv = p.z[om + i];
            const double d = sqrt(sv / zv);
            p.d[om + i] = d;
            const double di = 1.0 / d;
            p.di[om + i] = di;
            p.di2[om + i] = di * di;
            p.lmbda[om + i] = sqrt(sv * zv);
        }
        const double l = p.lmbda[om + i];
        p.lmbdasq[om + i] = l * l;
    }
    if (tid == 0) { S.mu = S.gap / (p.c.ml + p.c.nq); S.sigma = 0.0; S.eta = 0.0; }       // :2357-2358
}
// f4_no_ir's preamble for one cone (:2303-2309): s := lambda o\ s, z := z - W's, bzp := W^{-T} z for the solve
template <class Gp>
__device__ void q_f4_pre(const Gp &g, const Ptrs &p, long long oq, const double *v, double beta, int mq,
                         double *zv, double *sv, double *sh) {
    q_sinv(g, sv + oq, p.lmbda + oq, mq, sh);
    for (int j = g.rank(); j < mq; j += g.size()) p.bzp[oq + j] = sv[oq + j];
    g.sync();
    q_scale(g, p.bzp + oq, v, beta, mq, false, sh);                  // W' = W for 'q'
    for (int j = g.rank(); j < mq; j += g.size()) {
        const double t = zv[oq + j] - p.bzp[oq + j];
        zv[oq + j] = t;
        p.bzp[oq + j] = t;
    }
    g.sync();
    q_scale(g, p.bzp + oq, v, beta, mq, true, sh);
}
// right-hand side of the i-th Newton system and the f4_no_ir preamble (:2376-2309); save: keep the right-hand side
// for iterative refinement (f4, :2330-2336)
template <class Gp>
__global__ void k_dir_prep(Ptrs p, int i, int save) {
    PB_SETUP
    const double sm = S.sigma * S.mu, c = -1.0 + S.eta;
    for (int k = tid; k < p.n; k += nt) {
        const double v = c * p.rx[on + k];
        p.dx[on + k] = v;
        if (save) p.wx[on + k] = v;
    }
    const long long op = (long long)b * p.neq;
    for (int k = tid; k < p.neq; k += nt) {
        const double v = c * p.ry[op + k];
        p.dy[op + k] = v;
        if (save) p.wy[op + k] = v;
    }
    for (int k = tid; k < p.c.ml; k += nt) {
        double ds = -p.lmbdasq[om + k] + sm;
        if (i == 1) ds -= p.ws3[om + k];                 // Mehrotra correction
        if (save) { p.ws[om + k] = ds; p.wz[om + k] = c * p.rz[om + k]; }
        ds = ds / p.lmbda[om + k];                       // sinv
        p.ds[om + k] = ds;
        const double dz = c * p.rz[om + k] - p.d[om + k] * ds;   // z := z - W' s
        p.dz[om + k] = dz;
        p.bzp[om + k] = p.di[om + k] * dz;               // W^{-T} bz for the solve
    }
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k)
            for (int j = g.rank(); j < mq; j += g.size()) {
                // ds = -lambda o lambda (- ws3) + sigma mu e  (:2376-2385)
                double ds = -p.lmbdasq[oq + j] + sm * p.c.e[p.c.off[k] + j];
                if (i == 1) ds -= p.ws3[oq + j];
                const double bz = c * p.rz[oq + j];
                p.ds[oq + j] = ds;
                p.dz[oq + j] = bz;
                if (save) { p.ws[oq + j] = ds; p.wz[oq + j] = bz; }
            }
            g.sync();
            q_f4_pre(g, p, oq, vq_, *betaq_, mq, p.dz, p.ds, sh);
        }
    }
}
// refinement: the preamble of f4_no_ir on the correction's right-hand side (z2, s2)
template <class Gp>
__global__ void k_f4_pre(Ptrs p) {
    PB_SETUP
    (void)on; (void)S;
    for (int k = tid; k < p.c.ml; k += nt) {
        const double s = p.s2[om + k] / p.lmbda[om + k];
        p.s2[om + k] = s;
        const double z = p.z2[om + k] - p.d[om + k] * s;
        p.z2[om + k] = z;
        p.bzp[om + k] = p.di[om + k] * z;
    }
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k)
            q_f4_pre(g, p, oq, vq_, *betaq_, mq, p.z2, p.s2, sh);
        }
    }
}
// refinement: f4_no_ir's end (:2316) for the first solution: dz := uz (bzp), ds := ds - dz
__global__ void k_f4_post(Ptrs p) {
    PB_SETUP
    (void)sh; (void)S; (void)on;
    for (int k = tid; k < p.m; k += nt) {
        const double dz = p.bzp[om + k];
        p.dz[om + k] = dz;
        p.ds[om + k] -= dz;
    }
}
// refinement, res() (:1930-1960):  x2 = wx, y2 = wy (the GEMVs subtract P dx + A'dy + G'W^{-1}dz and A dx),
// t3 = W^{-1} dz,  z2 = wz - W'ds (the GEMV subtracts G dx),  s2 = ws - lambda o (dz + ds)
template <class Gp>
__global__ void k_res_prep(Ptrs p) {
    PB_SETUP
    (void)S;
    for (int k = tid; k < p.n; k += nt) p.x2[on + k] = p.wx[on + k];
    const long long op = (long long)b * p.neq;
    for (int k = tid; k < p.neq; k += nt) p.y2[op + k] = p.wy[op + k];
    for (int k = tid; k < p.c.ml; k += nt) {
        const double uz = p.dz[om + k], us = p.ds[om + k];
        p.t3[om + k] = p.di[om + k] * uz;
        p.z2[om + k] = p.wz[om + k] - p.d[om + k] * us;
        p.s2[om + k] = p.ws[om + k] - p.lmbda[om + k] * (us + uz);
    }
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k)
            for (int j = g.rank(); j < mq; j += g.size()) {
                const double uz = p.dz[oq + j], us = p.ds[oq + j];
                p.t3[oq + j] = uz; p.z2[oq + j] = us; p.s2[oq + j] = us + uz;
            }
            g.sync();
            q_scale(g, p.t3 + oq, vq_, *betaq_, mq, true, sh);
            q_scale(g, p.z2 + oq, vq_, *betaq_, mq, false, sh);
            q_sprod(g, p.s2 + oq, p.lmbda + oq, mq, sh);          // sprod(.., diag='D') is the same for 'q'
            for (int j = g.rank(); j < mq; j += g.size()) {
                p.z2[oq + j] = p.wz[oq + j] - p.z2[oq + j];
                p.s2[oq + j] = p.ws[oq + j] - p.s2[oq + j];
            }
            g.sync();
        }
    }
}
// refinement: dx += x2, dy += y2, dz += uz2, ds += s2 - uz2  (:2343-2347 after f4_no_ir's :2316)
__global__ void k_ref_add(Ptrs p) {
    PB_SETUP
    (void)sh; (void)S;
    for (int k = tid; k < p.n; k += nt) p.dx[on + k] += p.x2[on + k];
    const long long op = (long long)b * p.neq;
    for (int k = tid; k < p.neq; k += nt) p.dy[op + k] += p.y2[op + k];
    for (int k = tid; k < p.m; k += nt) {
        const double uz = p.bzp[om + k];
        p.dz[om + k] += uz;
        p.ds[om + k] += p.s2[om + k] - uz;
    }
}
// after the solve: dz = bzp (= W uz); ds := ds - dz (done already when refined); step length, sigma
// (:2316, :2423-2456)
template <class Gp>
__global__ void k_dir_post(Ptrs p, int i, int refined) {
    PB_SETUP
    double dsdz = 0, mins = INFINITY, minz = INFINITY;
    double tq = -INFINITY;                               // max_step over the cones
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k) (void)vq_; (void)betaq_;
            for (int j = g.rank(); j < mq; j += g.size()) {
                const double dz = refined ? p.dz[oq + j] : p.bzp[oq + j];
                const double ds = refined ? p.ds[oq + j] : p.ds[oq + j] - dz;
                p.dz[oq + j] = dz; p.ds[oq + j] = ds;
                dsdz += ds * dz;
                if (i == 0) p.ws3[oq + j] = ds;
            }
            g.sync();
            if (i == 0) q_sprod(g, p.ws3 + oq, p.dz + oq, mq, sh);   // ws3 = ds o dz (:2426-2428)
            q_scale2(g, p.lmbda + oq, p.ds + oq, mq, false, sh);
            q_scale2(g, p.lmbda + oq, p.dz + oq, mq, false, sh);
            const double t1 = q_max_step(g, p.ds + oq, mq, sh);
            const double t2 = q_max_step(g, p.dz + oq, mq, sh);
            tq = fmax(tq, fmax(t1, t2));
        }
    }
    for (int k = tid; k < p.c.ml; k += nt) {
        const double dz = refined ? p.dz[om + k] : p.bzp[om + k];
        const double ds = refined ? p.ds[om + k] : p.ds[om + k] - dz;
        dsdz += ds * dz;
        if (i == 0) p.ws3[om + k] = ds * dz;
        const double l = p.lmbda[om + k];
        const double dss = ds / l, dzs = dz / l;        // scale2
        p.ds[om + k] = dss; p.dz[om + k] = dzs;
        mins = fmin(mins, dss); minz = fmin(minz, dzs);
    }
    dsdz = block_sum(dsdz, sh);
    mins = block_min(mins, sh);
    minz = block_min(minz, sh);
    if (p.c.nq > 0) tq = block_max(tq, sh);
    if (tid == 0) {
        double t = fmax(0.0, fmax(-mins, -minz));
        if (p.c.nq > 0) t = fmax(t, tq);
        double step;
        if (t == 0.0) step = 1.0;
        else step = (i == 0) ? fmin(1.0, 1.0 / t) : fmin(1.0, 0.99 / t);
        S.step = step; S.dsdz = dsdz;
        if (i == 0) {
            const double v = fmin(1.0, fmax(0.0, 1.0 - step + dsdz / S.gap * step * step));
            S.sigma = v * v * v;
            S.eta = 0.0;
        }
    }
}
// x += step dx; new scaled iterates, scaling update, unscaled s, z, gap (:2459-2547, misc.py:450-464, 'q': :504-573)
template <class Gp>
__global__ void k_update(Ptrs p, const int *info, int iter) {
    PB_SETUP
    if (S.done) return;
    if (info[b] > 0) {      // non-positive pivot: "Terminated (singular KKT matrix)" (:2257-2275)
        if (tid == 0) { S.done = 1; S.status = 3; S.iters = iter; }
        return;
    }
    const double step = S.step;
    for (int k = tid; k < p.n; k += nt) p.x[on + k] += step * p.dx[on + k];
    const long long op = (long long)b * p.neq;
    for (int k = tid; k < p.neq; k += nt) p.y[op + k] += step * p.dy[op + k];
    double gap = 0;
    for (int k = tid; k < p.c.ml; k += nt) {
        const double l = p.lmbda[om + k];
        const double ds = (1.0 + step * p.ds[om + k]) * l;      // scale2 inverse
        const double dz = (1.0 + step * p.dz[om + k]) * l;
        const double ss = sqrt(ds), sz = sqrt(dz);
        const double d = p.d[om + k] * ss / sz;
        const double di = 1.0 / d;
        const double ln = ss * sz;
        p.d[om + k] = d; p.di[om + k] = di; p.di2[om + k] = di * di;
        p.lmbda[om + k] = ln;
        p.s[om + k] = d * ln;                                   // W' lambda
        p.z[om + k] = di * ln;                                  // W^{-1} lambda
        gap += ln * ln;
    }
    if (p.c.nq > 0) {
        const Gp g;
        Q_LOOP(g) {
            Q_CONE(k)
            const double *e = p.c.e + p.c.off[k];
            for (int j = g.rank(); j < mq; j += g.size()) {       // ds := e + step ds, dz := e + step dz
                p.ds[oq + j] = step * p.ds[oq + j] + e[j];
                p.dz[oq + j] = step * p.dz[oq + j] + e[j];
            }
            g.sync();
            q_scale2(g, p.lmbda + oq, p.ds + oq, mq, true, sh);
            q_scale2(g, p.lmbda + oq, p.dz + oq, mq, true, sh);
            q_update_scaling(g, p.ds + oq, p.dz + oq, vq_, betaq_, p.lmbda + oq, mq, sh);
            for (int j = g.rank(); j < mq; j += g.size()) {
                const double l = p.lmbda[oq + j];
                p.s[oq + j] = l; p.z[oq + j] = l;
                gap += l * l;
            }
            g.sync();
            q_scale(g, p.s + oq, vq_, *betaq_, mq, false, sh);      // s = W' lambda
            q_scale(g, p.z + oq, vq_, *betaq_, mq, true, sh);       // z = W^{-1} lambda
        }
    }
    gap = block_sum(gap, sh);
    if (tid == 0) S.gap = gap;
}

// Gs_q := W^{-T} G_q for every problem (blockIdx.y), column and cone: the 'q' rows of the scaled G whose Gram matrix
// enters S = P + G' W^{-1} W^{-T} G (kkt_chol2 / kkt_chol, misc.py:1407-1418).  Same arithmetic as scale_q_kernel
// (cone.cu) with inverse; W is symmetric.  One thread (cones of <= 8 rows) or one warp per (column, cone); cones
// vary fastest, so the threads of a warp read neighbouring rows of a column.
template <bool PerThread>
__global__ void k_scale_gq(Ptrs p, const double *G, long long ldg, long long sG, double *Gs, long long ldgs,
                           long long sGs) {
    constexpr int per = PerThread ? 1 : 32;
    const long long b = blockIdx.y;
    const long long item = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / per;
    const int lane = PerThread ? 0 : (threadIdx.x & 31);
    if (item >= (long long)p.n * p.c.nq) return;
    const int k = (int)(item % p.c.nq);
    const long long j = item / p.c.nq;
    const int mq = p.c.dim[k];
    const double *x = G + b * sG + j * ldg + p.c.ml + p.c.off[k];
    double *y = Gs + b * sGs + j * ldgs + p.c.off[k];
    const double *vb = p.c.vb + b * (p.c.sumq + p.c.nq);
    const double *v = vb + p.c.off[k];
    double w = 0;
    for (int i = lane; i < mq; i += per) w += v[i] * (i == 0 ? -x[i] : x[i]);
    if (!PerThread) w = warp_sum(w);
    const double tw = 2.0 * w, bi = 1.0 / vb[p.c.sumq + k];
    for (int i = lane; i < mq; i += per) {
        double yi = x[i] + v[i] * tw;
        if (i == 0) yi = -yi;
        y[i] = yi * bi;
    }
}

}  // namespace

struct cvxb_batch {
    int device = 0, B = 0, n = 0, m = 0;
    long long ldg = 0, ldp = 0, ldk = 0;
    long long sG = 0, sP = 0, sK = 0, sInv = 0;
    int nblk = 0;
    double *P = nullptr, *G = nullptr, *q = nullptr, *h = nullptr;
    // equality constraints A x = b (p = neq rows; nothing is allocated when p = 0)
    int neq = 0;
    long long lda = 0, ldkp = 0, sA = 0, sAs = 0, sKp = 0, sInvp = 0;
    double *A = nullptr;             // p x n per problem (ld lda)
    double *Asct = nullptr;          // n x p per problem (ld ldk): L^{-1} A'
    double *Kp = nullptr, *invp = nullptr;   // p x p per problem (ld ldkp): Asct' Asct, then its Cholesky factor
    double *veq = nullptr;           // p-vectors: b y ry dy wsing
    int *d_infop = nullptr, *d_nsing = nullptr;
    int nsing = 0;                   // problems flagged singular at the start of the last solve
    bool eq_loaded = false;
    // CVXB_BATCH_PHASE_MS=1 (read at create): time the factorisations' phases, synchronising after each one
    bool time_phases = false;
    double phase_ms[3] = {0, 0, 0};  // S: SYRK + Cholesky; TRSM (Asct); Kp: SYRK + Cholesky
    cudaEvent_t ph[4] = {nullptr, nullptr, nullptr, nullptr};
    double qphase_ms[2] = {0, 0};    // within S: the Gs_q scaling; the GEMM K += Gs_q' Gs_q
    cudaEvent_t qph[3] = {nullptr, nullptr, nullptr};
    // 'q' cones (dims = {'l': ml, 'q': qdim}; m = ml + sumq).  Nothing below is allocated without cones.
    int ml = 0, nq = 0, sumq = 0;
    int qmode = 0;                   // threads per cone in the cone kernels: 0 one, 1 a warp, 2 the CTA
    std::vector<int> qdim;
    int *d_qtab = nullptr;           // dim[nq], off[nq]
    double *qe = nullptr;            // sumq: the cones' identity e
    double *vb = nullptr;            // per problem: v (sumq), beta (nq)
    double *Gs = nullptr;            // per problem: W^{-T} G_q, sumq x n (ld ldgs)
    long long ldgs = 0, sGs = 0;
    // iterative refinement workspace, allocated by the first solve that refines
    double *refw = nullptr;
    double *K = nullptr, *inv = nullptr, *panel = nullptr, *gemv_ws = nullptr;
    double *vecs = nullptr;          // all n- and m-vectors
    Ptrs p;
    Scal *sc = nullptr;
    int *d_info = nullptr, *d_ndone = nullptr;
    int *d_done = nullptr, *d_pairs = nullptr, *d_perm = nullptr;     // compaction: done flags, swap list, slot -> problem
    std::vector<int> perm;           // slot -> original problem index (identity unless the last solve compacted)
    bool permuted = false;
    int compact = 1;                 // CVXB_BATCH_COMPACT=0 disables
    int Bact = 0;                    // slots [0, Bact) are launched by the lock-step loop
    CholWork cw;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool loaded = false;
    int iters_run = 0;
    double solve_ms = 0;
    // single large problem: SYRK on the int8 tensor path (ozaki_syrk.cu), same rule as cvxb_kkt_factor:
    // mode 1 (default) when B == 1, n >= 4096, m >= 8192; 2: whenever B == 1; 0: never.  CVXB_OZAKI (or the
    // older CVXB_OZAKI_IPM) = 0/1/2 read at create.
    int i8_mode = 1;
    int syrk_path = 0;
    void *oz_work = nullptr;
    size_t oz_bytes = 0;
};

namespace {

void phase_mark(cvxb_batch *b, int k) {
    if (b->time_phases) cudaEventRecord(b->ph[k], b->st);
}
// adds the time between marks k and k+1 to phase k (synchronises: timing runs only)
void phase_add(cvxb_batch *b, int k) {
    if (!b->time_phases) return;
    float t = 0;
    cudaEventSynchronize(b->ph[k + 1]);
    if (cudaEventElapsedTime(&t, b->ph[k], b->ph[k + 1]) == cudaSuccess) b->phase_ms[k] += t;
    cudaGetLastError();
}

void qphase(cvxb_batch *b, int k) {
    if (b->time_phases) cudaEventRecord(b->qph[k], b->st);
}

// launch a cone kernel with the batch's group size per cone (GThread / GWarp / GBlock)
#define QLAUNCH(kern, grid, T, st, ...) do {                                         \
        switch (b->qmode) {                                                          \
        case 1: kern<GWarp><<<(grid), (T), 0, (st)>>>(__VA_ARGS__); break;           \
        case 2: kern<GBlock><<<(grid), (T), 0, (st)>>>(__VA_ARGS__); break;          \
        default: kern<GThread><<<(grid), (T), 0, (st)>>>(__VA_ARGS__); break;        \
        }                                                                            \
        count_launch();                                                              \
    } while (0)

// K := P + G_l' diag(di)^2 G_l + Gs_q' Gs_q (+ A' diag(wsing) A where flagged) and its Cholesky factor;
// d_info per problem
int factor_S(cvxb_batch *b, bool i8) {
    cudaStream_t st = b->st;
    if (i8) {
        CVXB_TRY(ozaki_syrk(b->n, b->ml, b->G, b->ldg, b->p.di, b->P, b->ldp, 1.0, b->K, b->ldk, 9, 0,
                            b->oz_work, nullptr, st));
    } else if (b->ml > 0 || b->nq == 0) {
        GemmDesc g;
        g.M = b->n; g.N = b->n; g.K = b->ml;
        g.X = b->G; g.ldx = (int)b->ldg; g.x_kmajor = true; g.sX = b->sG;
        g.Y = b->G; g.ldy = (int)b->ldg; g.y_kmajor = true; g.sY = b->sG;
        g.w = b->p.di2; g.sW = b->m;
        g.D = b->P; g.ldd = (int)b->ldp; g.sD = b->sP; g.beta = 1.0;
        g.C = b->K; g.ldc = (int)b->ldk; g.sC = b->sK;
        g.lower_only = true; g.batch = b->Bact;
        if (b->B == 1) g.splitk_ws = b->cw.splitk_ws;
        CVXB_TRY(dmma_gemm(g, st));
    }
    if (b->nq > 0) {
        // Gs_q = W^{-T} G_q, then K += Gs_q' Gs_q (K := P + Gs_q' Gs_q without 'l' rows), as cvxb_kkt_factor does
        // for its non-'l' rows
        qphase(b, 0);
        const bool per_thread = b->qmode == 0;
        const long long items = (long long)b->n * b->nq, per_block = per_thread ? 256 : 8;
        const dim3 grid((unsigned)((items + per_block - 1) / per_block), (unsigned)b->Bact);
        if (per_thread) k_scale_gq<true><<<grid, 256, 0, st>>>(b->p, b->G, b->ldg, b->sG, b->Gs, b->ldgs, b->sGs);
        else k_scale_gq<false><<<grid, 256, 0, st>>>(b->p, b->G, b->ldg, b->sG, b->Gs, b->ldgs, b->sGs);
        count_launch();
        CVXB_LAUNCH_CHECK();
        qphase(b, 1);
        GemmDesc g;
        g.M = b->n; g.N = b->n; g.K = b->sumq;
        g.X = b->Gs; g.ldx = (int)b->ldgs; g.x_kmajor = true; g.sX = b->sGs;
        g.Y = b->Gs; g.ldy = (int)b->ldgs; g.y_kmajor = true; g.sY = b->sGs;
        if (b->ml > 0 || i8) { g.D = b->K; g.ldd = (int)b->ldk; g.sD = b->sK; }
        else { g.D = b->P; g.ldd = (int)b->ldp; g.sD = b->sP; }
        g.beta = 1.0;
        g.C = b->K; g.ldc = (int)b->ldk; g.sC = b->sK;
        g.lower_only = true; g.batch = b->Bact;
        CVXB_TRY(dmma_gemm(g, st));
        qphase(b, 2);
        if (b->time_phases) {
            float t = 0;
            cudaEventSynchronize(b->qph[2]);
            if (cudaEventElapsedTime(&t, b->qph[0], b->qph[1]) == cudaSuccess) b->qphase_ms[0] += t;
            if (cudaEventElapsedTime(&t, b->qph[1], b->qph[2]) == cudaSuccess) b->qphase_ms[1] += t;
            cudaGetLastError();
        }
    }
    if (b->nsing > 0) {
        // K += A' diag(wsing) A: adds A'A to the flagged problems' S and exactly zero to the others (misc.py:1452-1454)
        GemmDesc g;
        g.M = b->n; g.N = b->n; g.K = b->neq;
        g.X = b->A; g.ldx = (int)b->lda; g.x_kmajor = true; g.sX = b->sA;
        g.Y = b->A; g.ldy = (int)b->lda; g.y_kmajor = true; g.sY = b->sA;
        g.w = b->p.wsing; g.sW = b->neq;
        g.D = b->K; g.ldd = (int)b->ldk; g.sD = b->sK; g.beta = 1.0;
        g.C = b->K; g.ldc = (int)b->ldk; g.sC = b->sK;
        g.lower_only = true; g.batch = b->Bact;
        CVXB_TRY(dmma_gemm(g, st));
    }
    if (b->B == 1) {
        CVXB_TRY(potrf_lower(b->n, b->K, (int)b->ldk, b->inv, b->cw, st));
        CVXB_CUDA(cudaMemcpyAsync(b->d_info, b->cw.d_info, sizeof(int), cudaMemcpyDeviceToDevice, st));
    } else {
        CVXB_TRY(potrf_lower_batched(b->n, b->K, (int)b->ldk, b->sK, b->inv, b->sInv, b->Bact, b->d_info,
                                     b->panel, (b->n + 1) & ~1, st));
    }
    return 0;
}

// Asct := L^{-1} A',  Kp := Asct' Asct = Lp Lp'  (misc.py:1464-1472); a failed Kp pivot is folded into d_info
int factor_eq(cvxb_batch *b) {
    cudaStream_t st = b->st;
    const int n = b->n, pe = b->neq, B = b->Bact;
    phase_mark(b, 1);
    {
        const long long tot = (long long)n * pe;
        const unsigned gx = (unsigned)((tot + 255) / 256 < 64 ? (tot + 255) / 256 : 64);
        k_transpose_A<<<dim3(gx, B), 256, 0, st>>>(b->A, b->lda, b->sA, b->Asct, b->ldk, b->sAs, n, pe);
        count_launch();
    }
    CVXB_TRY(trsm_lower_left(n, b->K, b->ldk, b->inv, b->Asct, b->ldk, pe, st, B, b->sK, b->sInv, b->sAs));
    phase_mark(b, 2);
    GemmDesc g;
    g.M = pe; g.N = pe; g.K = n;
    g.X = b->Asct; g.ldx = (int)b->ldk; g.x_kmajor = true; g.sX = b->sAs;
    g.Y = b->Asct; g.ldy = (int)b->ldk; g.y_kmajor = true; g.sY = b->sAs;
    g.C = b->Kp; g.ldc = (int)b->ldkp; g.sC = b->sKp;
    g.lower_only = true; g.batch = B;
    CVXB_TRY(dmma_gemm(g, st));
    CVXB_TRY(potrf_lower_batched(pe, b->Kp, (int)b->ldkp, b->sKp, b->invp, b->sInvp, B, b->d_infop, b->panel,
                                 (int)b->ldkp, st));
    k_fold_info<<<(B + 255) / 256, 256, 0, st>>>(b->d_infop, b->d_info, n, B);
    count_launch();
    CVXB_LAUNCH_CHECK();
    phase_mark(b, 3);
    phase_add(b, 1);
    phase_add(b, 2);
    return 0;
}

// first: the factorisation at the starting point (W = I), where kkt_chol2 decides which problems are singular
int batch_factor(cvxb_batch *b, bool first = false) {
    bool i8 = b->B == 1 && b->ml > 0 && (b->i8_mode == 2 || (b->i8_mode == 1 && b->n >= 4096 && b->ml >= 8192));
    if (i8) {
        // K = P + G_l' diag(di)^2 G_l from nine int8 slices per entry (fp64-accurate, ~1.8x the DMMA SYRK);
        // same size rule and same fallback (workspace does not fit -> DMMA kernel) as cvxb_kkt_factor
        const size_t need = ozaki_workspace_bytes(b->n, b->ml, 9);
        if (need > b->oz_bytes) {
            if (b->oz_work) cudaFree(b->oz_work);
            b->oz_work = nullptr; b->oz_bytes = 0;
            cudaError_t ae = cudaMalloc(&b->oz_work, need);
            if (ae == cudaErrorMemoryAllocation) { cudaGetLastError(); tmp_cache_release(); ae = cudaMalloc(&b->oz_work, need); }
            if (ae != cudaSuccess) {
                cudaGetLastError();
                b->oz_work = nullptr;
                i8 = false;
            } else {
                b->oz_bytes = need;
            }
        }
    }
    b->syrk_path = i8 ? 2 : 1;
    phase_mark(b, 0);
    CVXB_TRY(factor_S(b, i8));
    if (b->neq > 0 && first) {
        CVXB_CUDA(cudaMemsetAsync(b->d_nsing, 0, sizeof(int), b->st));
        k_flag_singular<<<b->Bact, 128, 0, b->st>>>(b->p, b->d_info, b->d_nsing);
        count_launch();
        CVXB_CUDA(cudaMemcpyAsync(&b->nsing, b->d_nsing, sizeof(int), cudaMemcpyDeviceToHost, b->st));
        CVXB_CUDA(cudaStreamSynchronize(b->st));
        if (b->nsing > 0) CVXB_TRY(factor_S(b, i8));
    }
    phase_mark(b, 1);
    phase_add(b, 0);
    if (b->neq > 0) CVXB_TRY(factor_eq(b));
    return 0;
}

// (x, y, bzp) := solution of the reduced KKT system; on entry x = bx, y = by, bzp = W^{-T} bz
int batch_solve(cvxb_batch *b, double *x, double *y) {
    cudaStream_t st = b->st;
    const int n = b->n, m = b->m, B = b->Bact, pe = b->neq, ml = b->ml;
    double *bzq = b->p.bzp + ml;                 // the 'q' rows of bzp
    GemvBatch gt; gt.batch = B; gt.sA = b->sG; gt.sw = m; gt.sx = m; gt.sy = n;
    // x := x + G_l' (di .* bzp_l) + Gs_q' bzp_q
    if (ml > 0 || b->nq == 0) CVXB_TRY(gemv_t(ml, n, b->G, b->ldg, b->p.di, b->p.bzp, 1.0, 1.0, x, st, gt));
    if (b->nq > 0) {
        GemvBatch gq; gq.batch = B; gq.sA = b->sGs; gq.sx = m; gq.sy = n;
        CVXB_TRY(gemv_t(b->sumq, n, b->Gs, b->ldgs, nullptr, bzq, 1.0, 1.0, x, st, gq));
    }
    if (pe == 0) {
        CVXB_TRY(potrs_lower(n, b->K, (int)b->ldk, b->inv, x, b->cw, st, B, b->sK, b->sInv, n));
    } else {
        // kkt_chol2's solve (misc.py:1526-1558)
        if (b->nsing > 0) {       // x += A' by where S + A'A is factored
            GemvBatch ga; ga.batch = B; ga.sA = b->sA; ga.sw = pe; ga.sx = pe; ga.sy = n;
            CVXB_TRY(gemv_t(pe, n, b->A, b->lda, b->p.wsing, y, 1.0, 1.0, x, st, ga));
        }
        CVXB_TRY(trsv_lower(n, b->K, (int)b->ldk, b->inv, x, false, b->cw, st, B, b->sK, b->sInv, n));
        GemvBatch gyt; gyt.batch = B; gyt.sA = b->sAs; gyt.sx = n; gyt.sy = pe;       // y := Asct' x - y
        CVXB_TRY(gemv_t(n, pe, b->Asct, b->ldk, nullptr, x, 1.0, -1.0, y, st, gyt));
        CVXB_TRY(potrs_lower(pe, b->Kp, (int)b->ldkp, b->invp, y, b->cw, st, B, b->sKp, b->sInvp, pe));
        GemvBatch gyn; gyn.batch = B; gyn.sA = b->sAs; gyn.sx = pe; gyn.sy = n;       // x -= Asct y
        CVXB_TRY(gemv_n(n, pe, b->Asct, b->ldk, nullptr, y, -1.0, 1.0, x, b->gemv_ws, st, gyn));
        CVXB_TRY(trsv_lower(n, b->K, (int)b->ldk, b->inv, x, true, b->cw, st, B, b->sK, b->sInv, n));
    }
    // bzp := [di .* (G_l x); Gs_q x] - bzp
    GemvBatch gn; gn.batch = B; gn.sA = b->sG; gn.sw = m; gn.sx = n; gn.sy = m;
    if (ml > 0 || b->nq == 0)
        CVXB_TRY(gemv_n(ml, n, b->G, b->ldg, b->p.di, x, 1.0, -1.0, b->p.bzp, b->gemv_ws, st, gn));
    if (b->nq > 0) {
        GemvBatch gq; gq.batch = B; gq.sA = b->sGs; gq.sx = n; gq.sy = m;
        CVXB_TRY(gemv_n(b->sumq, n, b->Gs, b->ldgs, nullptr, x, 1.0, -1.0, bzq, b->gemv_ws, st, gq));
    }
    return 0;
}

}  // namespace

extern "C" {

int cvxb_batch_create(cvxb_batch **out, int nprob, int n, int m, int device) {
    return cvxb_batch_create_eq(out, nprob, n, m, 0, device);
}

int cvxb_batch_create_eq(cvxb_batch **out, int nprob, int n, int m, int p, int device) {
    return cvxb_batch_create_cones(out, nprob, n, m, 0, nullptr, p, device);
}

int cvxb_batch_create_cones(cvxb_batch **out, int nprob, int n, int ml, int nq, const int *qdims, int p, int device) {
    if (!out || nprob <= 0 || n <= 0 || ml < 0) { set_error("batch_create: bad sizes"); return CVXB_E_ARG; }
    if (nq < 0 || (nq > 0 && !qdims)) { set_error("batch_create: bad 'q' cone list"); return CVXB_E_ARG; }
    long long msum = ml;
    int qmax = 0;
    for (int k = 0; k < nq; ++k) {
        if (qdims[k] < 1) { set_error("batch_create: 'q' cone %d has size %d (must be >= 1)", k, qdims[k]); return CVXB_E_ARG; }
        msum += qdims[k];
        qmax = std::max(qmax, qdims[k]);
    }
    if (msum > (1 << 30)) { set_error("batch_create: bad sizes"); return CVXB_E_ARG; }
    const int m = (int)msum;
    if (p < 0 || p > n) { set_error("batch_create: need 0 <= p <= n (p = %d, n = %d)", p, n); return CVXB_E_ARG; }
    if (p > 0 && m == 0) { set_error("batch_create: equality constraints need m > 0"); return CVXB_E_ARG; }
    *out = nullptr;
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        set_error("no CUDA device available: cvxopt_b200 has no CPU fallback");
        return CVXB_E_NOGPU;
    }
    if (device < 0 || device >= cnt) { set_error("device out of range"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(device));
    cvxb_batch *b = new cvxb_batch();
    b->device = device; b->B = nprob; b->n = n; b->m = m; b->neq = p;
    b->ml = ml; b->nq = nq; b->sumq = m - ml;
    b->qdim.assign(qdims, qdims + nq);
    // one thread per cone for cones of <= 8 rows, a warp per cone when there are enough of them to fill the CTA,
    // else the whole CTA per cone (a few large cones)
    b->qmode = qmax <= 8 ? 0 : (nq >= 256 / 32 ? 1 : 2);
    if (const char *e = getenv("CVXB_OZAKI")) b->i8_mode = (e[0] == '0') ? 0 : (e[0] == '2') ? 2 : 1;
    if (const char *e = getenv("CVXB_OZAKI_IPM")) b->i8_mode = (e[0] == '1') ? 1 : (e[0] == '2') ? 2 : 0;
    b->ldg = ((m + 1) & ~1) > 2 ? ((m + 1) & ~1) : 2;
    b->ldp = b->ldk = (n + 1) & ~1;
    b->sG = b->ldg * n; b->sP = b->ldp * n; b->sK = b->ldk * n;
    b->nblk = (n + NB - 1) / NB;
    b->sInv = (long long)2 * b->nblk * NB * NB;
    auto fail = [&](int r) { cvxb_batch_destroy(b); return r; };
#define BCUDA(expr) do { cudaError_t _e = (expr); \
        /* out of memory: give the scratch-buffer cache (common.cuh) back to the driver and try once more */ \
        if (_e == cudaErrorMemoryAllocation) { cudaGetLastError(); tmp_cache_release(); _e = (expr); } \
        if (_e != cudaSuccess) { \
        set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
        return fail(_e == cudaErrorMemoryAllocation ? CVXB_E_NOMEM : CVXB_E_CUDA); } } while (0)
    const size_t B = nprob;
    BCUDA(cudaStreamCreateWithFlags(&b->st, cudaStreamNonBlocking));
    BCUDA(cudaEventCreate(&b->e0)); BCUDA(cudaEventCreate(&b->e1));
    { int r = chol_work_create(b->cw); if (r) return fail(r); }
    BCUDA(cudaMalloc(&b->P, B * b->sP * sizeof(double)));
    BCUDA(cudaMalloc(&b->G, B * b->sG * sizeof(double)));
    BCUDA(cudaMalloc(&b->K, B * b->sK * sizeof(double)));
    BCUDA(cudaMalloc(&b->inv, B * b->sInv * sizeof(double)));
    BCUDA(cudaMalloc(&b->panel, B * (size_t)((n + 1) & ~1) * NB * sizeof(double)));
    {   // gemv_n workspace: rows of G, and with p > 0 also the n rows of Asct
        const size_t rows = (size_t)std::max(std::max(m, p > 0 ? n : 0), 1);
        BCUDA(cudaMalloc(&b->gemv_ws, B * rows * gemv_n_chunks(n) * sizeof(double)));
    }
    // vectors: n-sized: q x rx dx ; m-sized: h s z rz ds dz lmbda lmbdasq d di di2 ws3 bzp
    const size_t nv = 4, mv = 13;
    const size_t me = (size_t)(m > 0 ? m : 1);
    BCUDA(cudaMalloc(&b->vecs, B * (nv * n + mv * me) * sizeof(double)));
    BCUDA(cudaMemset(b->vecs, 0, B * (nv * n + mv * me) * sizeof(double)));
    double *v = b->vecs;
    auto take = [&](size_t len) { double *r = v; v += B * len; return r; };
    b->q = take(n); b->p.x = take(n); b->p.rx = take(n); b->p.dx = take(n);
    b->h = take(me); b->p.s = take(me); b->p.z = take(me); b->p.rz = take(me); b->p.ds = take(me);
    b->p.dz = take(me); b->p.lmbda = take(me); b->p.lmbdasq = take(me); b->p.d = take(me);
    b->p.di = take(me); b->p.di2 = take(me); b->p.ws3 = take(me); b->p.bzp = take(me);
    b->p.q = b->q; b->p.h = b->h; b->p.n = n; b->p.m = m;
    b->p.neq = p; b->p.beq = nullptr; b->p.y = b->p.ry = b->p.dy = b->p.wsing = nullptr;
    b->p.wx = b->p.wy = b->p.wz = b->p.ws = b->p.x2 = b->p.y2 = b->p.z2 = b->p.s2 = b->p.t3 = nullptr;
    b->p.c.ml = ml; b->p.c.nq = nq; b->p.c.sumq = b->sumq;
    b->p.c.dim = b->p.c.off = nullptr; b->p.c.e = nullptr; b->p.c.vb = nullptr;
    if (nq > 0) {
        std::vector<int> tab(2 * (size_t)nq);
        std::vector<double> e((size_t)b->sumq, 0.0);
        for (int k = 0, o = 0; k < nq; o += qdims[k], ++k) { tab[k] = qdims[k]; tab[nq + k] = o; e[o] = 1.0; }
        BCUDA(cudaMalloc(&b->d_qtab, tab.size() * sizeof(int)));
        BCUDA(cudaMemcpy(b->d_qtab, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice));
        BCUDA(cudaMalloc(&b->qe, e.size() * sizeof(double)));
        BCUDA(cudaMemcpy(b->qe, e.data(), e.size() * sizeof(double), cudaMemcpyHostToDevice));
        BCUDA(cudaMalloc(&b->vb, B * (size_t)(b->sumq + nq) * sizeof(double)));
        BCUDA(cudaMemset(b->vb, 0, B * (size_t)(b->sumq + nq) * sizeof(double)));
        b->ldgs = std::max<long long>(2, (b->sumq + 1) & ~1);
        b->sGs = b->ldgs * n;
        BCUDA(cudaMalloc(&b->Gs, B * b->sGs * sizeof(double)));
        b->p.c.dim = b->d_qtab; b->p.c.off = b->d_qtab + nq; b->p.c.e = b->qe; b->p.c.vb = b->vb;
    }
    if (p > 0) {
        b->lda = b->ldkp = (p + 1) & ~1;
        b->sA = b->lda * n; b->sAs = b->ldk * p; b->sKp = b->ldkp * p;
        b->sInvp = (long long)2 * ((p + NB - 1) / NB) * NB * NB;
        BCUDA(cudaMalloc(&b->A, B * b->sA * sizeof(double)));
        BCUDA(cudaMalloc(&b->Asct, B * b->sAs * sizeof(double)));
        BCUDA(cudaMalloc(&b->Kp, B * b->sKp * sizeof(double)));
        BCUDA(cudaMalloc(&b->invp, B * b->sInvp * sizeof(double)));
        BCUDA(cudaMalloc(&b->veq, B * 5 * (size_t)p * sizeof(double)));
        BCUDA(cudaMemset(b->veq, 0, B * 5 * (size_t)p * sizeof(double)));
        BCUDA(cudaMalloc(&b->d_infop, B * sizeof(int)));
        BCUDA(cudaMalloc(&b->d_nsing, sizeof(int)));
        double *w = b->veq;
        b->p.beq = w; b->p.y = w + B * p; b->p.ry = w + 2 * B * p; b->p.dy = w + 3 * B * p; b->p.wsing = w + 4 * B * p;
    }
    if (const char *e = getenv("CVXB_BATCH_PHASE_MS")) b->time_phases = e[0] == '1';
    if (b->time_phases) {
        for (cudaEvent_t &e : b->ph) BCUDA(cudaEventCreate(&e));
        for (cudaEvent_t &e : b->qph) BCUDA(cudaEventCreate(&e));
    }
    BCUDA(cudaMalloc(&b->sc, B * sizeof(Scal)));
    BCUDA(cudaMemset(b->sc, 0, B * sizeof(Scal)));
    b->p.sc = b->sc;
    BCUDA(cudaMalloc(&b->d_info, B * sizeof(int)));
    BCUDA(cudaMalloc(&b->d_ndone, sizeof(int)));
    BCUDA(cudaMalloc(&b->d_done, B * sizeof(int)));
    BCUDA(cudaMalloc(&b->d_pairs, 2 * B * sizeof(int)));
    BCUDA(cudaMalloc(&b->d_perm, B * sizeof(int)));
    b->perm.resize(B);
    for (size_t i = 0; i < B; ++i) b->perm[i] = (int)i;
    if (const char *e = getenv("CVXB_BATCH_COMPACT")) b->compact = (e[0] == '0') ? 0 : 1;
#undef BCUDA
    *out = b;
    return 0;
}

void cvxb_batch_destroy(cvxb_batch *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->st) cudaStreamSynchronize(b->st);
    double *bufs[] = {b->P, b->G, b->K, b->inv, b->panel, b->gemv_ws, b->vecs, b->A, b->Asct, b->Kp, b->invp, b->veq,
                      b->qe, b->vb, b->Gs, b->refw};
    for (double *x : bufs) if (x) cudaFree(x);
    if (b->d_qtab) cudaFree(b->d_qtab);
    for (cudaEvent_t e : b->qph) if (e) cudaEventDestroy(e);
    if (b->d_infop) cudaFree(b->d_infop);
    if (b->d_nsing) cudaFree(b->d_nsing);
    for (cudaEvent_t e : b->ph) if (e) cudaEventDestroy(e);
    if (b->sc) cudaFree(b->sc);
    if (b->oz_work) cudaFree(b->oz_work);
    if (b->d_info) cudaFree(b->d_info);
    if (b->d_ndone) cudaFree(b->d_ndone);
    if (b->d_done) cudaFree(b->d_done);
    if (b->d_pairs) cudaFree(b->d_pairs);
    if (b->d_perm) cudaFree(b->d_perm);
    chol_work_destroy(b->cw);
    if (b->e0) cudaEventDestroy(b->e0);
    if (b->e1) cudaEventDestroy(b->e1);
    if (b->st) cudaStreamDestroy(b->st);
    delete b;
}

// P: nprob x (n x n, ld n) ; q: nprob x n ; G: nprob x (m x n column-major, ld m) ; h: nprob x m
int cvxb_batch_load(cvxb_batch *b, const double *P, const double *q, const double *G,
                    const double *h, int space) {
    if (!b || !P || !q || (b->m > 0 && (!G || !h))) { set_error("batch_load: NULL argument"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(b->device));
    const cudaMemcpyKind kind = (space == CVXB_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const size_t B = b->B, n = b->n, m = b->m;
    // one strided 2-D copy per operand: rows of the "matrix of columns" are the matrix columns
    CVXB_CUDA(cudaMemcpy2DAsync(b->P, b->ldp * sizeof(double), P, n * sizeof(double), n * sizeof(double),
                                n * B, kind, b->st));
    if (m > 0) {
        CVXB_CUDA(cudaMemcpy2DAsync(b->G, b->ldg * sizeof(double), G, m * sizeof(double),
                                    m * sizeof(double), n * B, kind, b->st));
        CVXB_CUDA(cudaMemcpyAsync(const_cast<double *>(b->h), h, B * m * sizeof(double), kind, b->st));
    }
    CVXB_CUDA(cudaMemcpyAsync(const_cast<double *>(b->q), q, B * n * sizeof(double), kind, b->st));
    // only tril(P) is significant in the reference; make the resident copies symmetric
    CVXB_TRY(symmetrize_lower(b->n, b->P, b->ldp, b->B, b->sP, b->st));
    CVXB_CUDA(cudaStreamSynchronize(b->st));
    b->loaded = true;
    b->eq_loaded = false;        // A and b are loaded after P, q, G, h (cvxb_batch_load_eq)
    for (size_t i = 0; i < B; ++i) b->perm[i] = (int)i;
    b->permuted = false;
    return 0;
}

// swap the slots of each pair (disjoint pairs: one launch)
static int swap_slots(cvxb_batch *b, const std::vector<int> &pairs) {
    const int np = (int)pairs.size() / 2;
    if (np == 0) return 0;
    CVXB_CUDA(cudaMemcpyAsync(b->d_pairs, pairs.data(), pairs.size() * sizeof(int), cudaMemcpyHostToDevice, b->st));
    SwapArgs a;
    a.P = b->P; a.G = b->G; a.vecs = b->vecs; a.sc = b->sc; a.sP = b->sP; a.sG = b->sG;
    a.n = b->n; a.me = b->m > 0 ? b->m : 1; a.Btot = b->B;
    a.A = b->A; a.veq = b->veq; a.sA = b->sA; a.neq = b->neq;
    a.vb = b->vb; a.nvb = b->nq > 0 ? b->sumq + b->nq : 0;
    k_swap_slots<<<dim3(96, np), 256, 0, b->st>>>(a, b->d_pairs);
    count_launch();
    // `pairs` is pageable host memory: the copy above is staged before cudaMemcpyAsync returns
    return 0;
}

// put every problem back into its own slot (a solve that compacted left them permuted)
static int restore_order(cvxb_batch *b) {
    if (!b->permuted) return 0;
    std::vector<int> pr(2);
    for (int i = 0; i < b->B; ++i) {
        while (b->perm[i] != i) {
            const int j = b->perm[i];                // the problem in slot i belongs to slot j
            pr[0] = i; pr[1] = j;
            CVXB_TRY(swap_slots(b, pr));
            std::swap(b->perm[i], b->perm[j]);
        }
    }
    CVXB_CUDA(cudaStreamSynchronize(b->st));
    b->permuted = false;
    return 0;
}

// A: nprob x (p x n column-major, ld p) ; bvec: nprob x p.  After cvxb_batch_load.
int cvxb_batch_load_eq(cvxb_batch *b, const double *A, const double *bvec, int space) {
    if (!b) { set_error("batch is NULL"); return CVXB_E_ARG; }
    if (!b->loaded) { set_error("batch_load_eq: call cvxb_batch_load first"); return CVXB_E_ARG; }
    if (b->neq == 0) { b->eq_loaded = true; return 0; }
    if (!A || !bvec) { set_error("batch_load_eq: NULL argument"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(b->device));
    CVXB_TRY(restore_order(b));
    const cudaMemcpyKind kind = (space == CVXB_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const size_t B = b->B, n = b->n, p = b->neq;
    CVXB_CUDA(cudaMemcpy2DAsync(b->A, b->lda * sizeof(double), A, p * sizeof(double), p * sizeof(double), n * B,
                                kind, b->st));
    CVXB_CUDA(cudaMemcpyAsync(const_cast<double *>(b->p.beq), bvec, B * p * sizeof(double), kind, b->st));
    CVXB_CUDA(cudaStreamSynchronize(b->st));
    b->eq_loaded = true;
    return 0;
}

int cvxb_batch_solve(cvxb_batch *b, int maxiters, double abstol, double reltol, double feastol) {
    return cvxb_batch_solve_ref(b, maxiters, abstol, reltol, feastol, -1);
}

int cvxb_batch_solve_ref(cvxb_batch *b, int maxiters, double abstol, double reltol, double feastol, int refinement) {
    if (!b || !b->loaded) { set_error("batch_solve: load the problems first"); return CVXB_E_ARG; }
    // coneqp's default: one step of iterative refinement when there are 'q' cones, none otherwise (:1862-1865)
    const int refine = refinement >= 0 ? refinement : (b->nq > 0 ? 1 : 0);
    if (b->neq > 0 && !b->eq_loaded) { set_error("batch_solve: load A and b (cvxb_batch_load_eq) first"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(b->device));
    cudaStream_t st = b->st;
    CVXB_TRY(restore_order(b));
    const int n = b->n, m = b->m, T = 256;
    if (refine > 0 && !b->refw) {
        // wx x2 (n), wy y2 (p), wz ws z2 s2 t3 (m) per problem
        const size_t per = 2 * (size_t)n + 2 * (size_t)b->neq + 5 * (size_t)m;
        cudaError_t e = cudaMalloc(&b->refw, (size_t)b->B * per * sizeof(double));
        if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); tmp_cache_release(); e = cudaMalloc(&b->refw, (size_t)b->B * per * sizeof(double)); }
        if (e != cudaSuccess) {
            cudaGetLastError();
            b->refw = nullptr;
            set_error("batch_solve: no memory for the refinement workspace");
            return e == cudaErrorMemoryAllocation ? CVXB_E_NOMEM : CVXB_E_CUDA;
        }
        double *w = b->refw;
        const size_t Bt = b->B;
        auto take = [&](size_t len) { double *r = w; w += Bt * len; return r; };
        Ptrs &q = b->p;
        q.wx = take(n); q.x2 = take(n); q.wy = take(b->neq); q.y2 = take(b->neq);
        q.wz = take(m); q.ws = take(m); q.z2 = take(m); q.s2 = take(m); q.t3 = take(m);
    }
    int B = b->B;                                 // active slots: shrinks as problems finish (compaction)
    b->Bact = B;
    Ptrs &p = b->p;
    GemvBatch gP; gP.batch = B; gP.sA = b->sP; gP.sx = n; gP.sy = n;
    GemvBatch gGt; gGt.batch = B; gGt.sA = b->sG; gGt.sx = m; gGt.sy = n;
    GemvBatch gGn; gGn.batch = B; gGn.sA = b->sG; gGn.sx = n; gGn.sy = m;
    CVXB_CUDA(cudaMemsetAsync(b->sc, 0, (size_t)B * sizeof(Scal), st));
    b->nsing = 0;
    if (b->neq > 0) CVXB_CUDA(cudaMemsetAsync(p.wsing, 0, (size_t)B * b->neq * sizeof(double), st));
    for (double &t : b->phase_ms) t = 0;
    for (double &t : b->qphase_ms) t = 0;
    GemvBatch gAt; gAt.batch = B; gAt.sA = b->sA; gAt.sx = b->neq; gAt.sy = n;
    GemvBatch gAn; gAn.batch = B; gAn.sA = b->sA; gAn.sx = n; gAn.sy = b->neq;
    CVXB_CUDA(cudaEventRecord(b->e0, st));
    // ---- starting point: W = I ----
    k_init_rhs<<<B, T, 0, st>>>(p); count_launch();
    CVXB_TRY(batch_factor(b, true));
    k_scale_bz<<<B, T, 0, st>>>(p, p.dz); count_launch();
    CVXB_TRY(batch_solve(b, p.dx, p.dy));
    QLAUNCH(k_init_point, B, T, st, p);
    CVXB_LAUNCH_CHECK();
    int info_fail = 0;
    {
        // a singular first factorisation is the reference's "Rank([P; G]) < n" ValueError
        std::vector<int> info(B);
        CVXB_CUDA(cudaMemcpyAsync(info.data(), b->d_info, B * sizeof(int), cudaMemcpyDeviceToHost, st));
        CVXB_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < B; ++i) if (info[i] > 0) { info_fail = i + 1; break; }
        if (info_fail) {
            if (b->neq > 0)
                set_error("batch_solve: problem %d: Rank(A) < p or Rank([P; A; G]) < n (singular KKT matrix at the "
                          "start)", info_fail - 1);
            else
                set_error("batch_solve: problem %d: Rank([P; G]) < n (singular KKT matrix at the start)", info_fail - 1);
            return CVXB_E_ARG;
        }
    }
    std::vector<int> flags(B), pairs;
    int it = 0;
    for (it = 0; it <= maxiters; ++it) {
        // residuals (:2169-2186)
        k_res_begin<<<B, T, 0, st>>>(p); count_launch();
        CVXB_TRY(gemv_t(n, n, b->P, b->ldp, nullptr, p.x, 1.0, 1.0, p.rx, st, gP));
        k_res_dots<<<B, T, 0, st>>>(p); count_launch();
        if (b->neq > 0) CVXB_TRY(gemv_t(b->neq, n, b->A, b->lda, nullptr, p.y, 1.0, 1.0, p.rx, st, gAt));   // rx += A'y
        if (m > 0) {
            CVXB_TRY(gemv_t(m, n, b->G, b->ldg, nullptr, p.z, 1.0, 1.0, p.rx, st, gGt));
            CVXB_TRY(gemv_n(m, n, b->G, b->ldg, nullptr, p.x, 1.0, 1.0, p.rz, b->gemv_ws, st, gGn));
        }
        if (b->neq > 0)        // ry := A x - b
            CVXB_TRY(gemv_n(b->neq, n, b->A, b->lda, nullptr, p.x, 1.0, -1.0, p.ry, b->gemv_ws, st, gAn));
        CVXB_CUDA(cudaMemsetAsync(b->d_ndone, 0, sizeof(int), st));
        k_stats<<<B, T, 0, st>>>(p, it, maxiters, abstol, reltol, feastol, b->d_ndone, b->d_done); count_launch();
        int ndone = 0;
        CVXB_CUDA(cudaMemcpyAsync(&ndone, b->d_ndone, sizeof(int), cudaMemcpyDeviceToHost, st));
        CVXB_CUDA(cudaMemcpyAsync(flags.data(), b->d_done, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
        CVXB_CUDA(cudaStreamSynchronize(st));
        if (ndone >= B) break;
        if (ndone > 0 && b->compact && b->B > 1) {
            // finished slots below the new active count trade places with active slots from the tail
            const int nb = B - ndone;
            pairs.clear();
            int j = B - 1;
            for (int i = 0; i < nb; ++i) {
                if (!flags[i]) continue;
                while (flags[j]) --j;             // an active slot in [nb, B): there are as many as finished ones below nb
                pairs.push_back(i); pairs.push_back(j);
                std::swap(b->perm[i], b->perm[j]);
                --j;
            }
            CVXB_TRY(swap_slots(b, pairs));
            b->permuted = true;
            B = nb;
            b->Bact = B;
            gP.batch = gGt.batch = gGn.batch = gAt.batch = gAn.batch = B;
        }
        QLAUNCH(k_scaling, B, T, st, p, it == 0 ? 1 : 0);
        CVXB_TRY(batch_factor(b));
        for (int i = 0; i < 2; ++i) {
            QLAUNCH(k_dir_prep, B, T, st, p, i, refine > 0 ? 1 : 0);
            CVXB_TRY(batch_solve(b, p.dx, p.dy));
            if (refine > 0) {
                // f4: refine the solution with the residual of the Newton system (:2330-2347)
                k_f4_post<<<B, T, 0, st>>>(p); count_launch();
                for (int r = 0; r < refine; ++r) {
                    QLAUNCH(k_res_prep, B, T, st, p);
                    CVXB_TRY(gemv_t(n, n, b->P, b->ldp, nullptr, p.dx, -1.0, 1.0, p.x2, st, gP));
                    if (b->neq > 0) {
                        CVXB_TRY(gemv_t(b->neq, n, b->A, b->lda, nullptr, p.dy, -1.0, 1.0, p.x2, st, gAt));
                        CVXB_TRY(gemv_n(b->neq, n, b->A, b->lda, nullptr, p.dx, -1.0, 1.0, p.y2, b->gemv_ws, st, gAn));
                    }
                    if (m > 0) {
                        CVXB_TRY(gemv_t(m, n, b->G, b->ldg, nullptr, p.t3, -1.0, 1.0, p.x2, st, gGt));
                        CVXB_TRY(gemv_n(m, n, b->G, b->ldg, nullptr, p.dx, -1.0, 1.0, p.z2, b->gemv_ws, st, gGn));
                    }
                    QLAUNCH(k_f4_pre, B, T, st, p);
                    CVXB_TRY(batch_solve(b, p.x2, p.y2));
                    k_ref_add<<<B, T, 0, st>>>(p); count_launch();
                }
            }
            QLAUNCH(k_dir_post, B, T, st, p, i, refine > 0 ? 1 : 0);
        }
        QLAUNCH(k_update, B, T, st, p, b->d_info, it);
        CVXB_LAUNCH_CHECK();
    }
    b->iters_run = it;
    b->Bact = b->B;
    CVXB_CUDA(cudaEventRecord(b->e1, st));
    CVXB_CUDA(cudaStreamSynchronize(st));
    float t = 0;
    cudaEventElapsedTime(&t, b->e0, b->e1);
    b->solve_ms = t;
    return 0;
}

// dst[problem, :len] = src[slot, :len] for every slot (rows of length len, one per problem)
static int give_rows(cvxb_batch *b, double *dst, const double *src, int len, int space) {
    const cudaMemcpyKind kind = (space == CVXB_DEVICE) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    const size_t B = b->B;
    if (!b->permuted) { CVXB_CUDA(cudaMemcpy(dst, src, B * len * sizeof(double), kind)); return 0; }
    // slot -> problem (identity unless the solve compacted finished problems away)
    CVXB_CUDA(cudaMemcpy(b->d_perm, b->perm.data(), B * sizeof(int), cudaMemcpyHostToDevice));
    double *tmp = (space == CVXB_DEVICE) ? dst : nullptr;
    if (!tmp) CVXB_CUDA(tmp_malloc(&tmp, B * len * sizeof(double)));
    k_unpermute_rows<<<(unsigned)B, 256, 0, b->st>>>(src, tmp, b->d_perm, len);
    count_launch();
    cudaError_t e = cudaStreamSynchronize(b->st);
    if (e == cudaSuccess && tmp != dst) e = cudaMemcpy(dst, tmp, B * len * sizeof(double), kind);
    if (tmp != dst) tmp_free(tmp);
    CVXB_CUDA(e);
    return 0;
}

int cvxb_batch_results(cvxb_batch *b, double *x, double *s, double *z, int *status, int *iters,
                       double *pobj, double *dobj, int space) {
    if (!b) { set_error("batch is NULL"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(b->device));
    const size_t B = b->B;
    auto give = [&](double *dst, const double *src, int len) { return give_rows(b, dst, src, len, space); };
    if (x) CVXB_TRY(give(x, b->p.x, b->n));
    if (s && b->m) CVXB_TRY(give(s, b->p.s, b->m));
    if (z && b->m) CVXB_TRY(give(z, b->p.z, b->m));
    if (status || iters || pobj || dobj) {
        if (space == CVXB_DEVICE) { set_error("batch_results: scalars are returned to host memory only"); return CVXB_E_ARG; }
        std::vector<Scal> sc(B);
        CVXB_CUDA(cudaMemcpy(sc.data(), b->sc, B * sizeof(Scal), cudaMemcpyDeviceToHost));
        for (size_t slot = 0; slot < B; ++slot) {
            const size_t i = (size_t)b->perm[slot];
            if (status) status[i] = sc[slot].status;
            if (iters) iters[i] = sc[slot].iters;
            if (pobj) pobj[i] = sc[slot].pcost;
            if (dobj) dobj[i] = sc[slot].dcost;
        }
    }
    return 0;
}

int cvxb_batch_results_y(cvxb_batch *b, double *y, int space) {
    if (!b || !y) { set_error("batch_results_y: NULL argument"); return CVXB_E_ARG; }
    if (b->neq == 0) return 0;
    CVXB_CUDA(cudaSetDevice(b->device));
    return give_rows(b, y, b->p.y, b->neq, space);
}

int cvxb_batch_singular(cvxb_batch *b, int *flags) {
    if (!b || !flags) { set_error("batch_singular: NULL argument"); return CVXB_E_ARG; }
    CVXB_CUDA(cudaSetDevice(b->device));
    std::vector<Scal> sc(b->B);
    CVXB_CUDA(cudaMemcpy(sc.data(), b->sc, sc.size() * sizeof(Scal), cudaMemcpyDeviceToHost));
    for (int slot = 0; slot < b->B; ++slot) flags[b->perm[slot]] = sc[slot].singular;
    return 0;
}

int cvxb_batch_phase_ms(cvxb_batch *b, double *ms) {
    if (!b || !ms) { set_error("batch_phase_ms: NULL argument"); return CVXB_E_ARG; }
    if (!b->time_phases) { set_error("batch_phase_ms: create the batch with CVXB_BATCH_PHASE_MS=1"); return CVXB_E_ARG; }
    for (int k = 0; k < 3; ++k) ms[k] = b->phase_ms[k];
    return 0;
}

int cvxb_batch_phase_ms_cones(cvxb_batch *b, double *ms) {
    if (!b || !ms) { set_error("batch_phase_ms_cones: NULL argument"); return CVXB_E_ARG; }
    if (!b->time_phases) { set_error("batch_phase_ms_cones: create the batch with CVXB_BATCH_PHASE_MS=1"); return CVXB_E_ARG; }
    for (int k = 0; k < 2; ++k) ms[k] = b->qphase_ms[k];
    return 0;
}

int cvxb_batch_syrk_path(cvxb_batch *b) { return b ? b->syrk_path : CVXB_E_ARG; }

int cvxb_batch_stats(cvxb_batch *b, double *solve_ms, int *iterations) {
    if (!b) return CVXB_E_ARG;
    if (solve_ms) *solve_ms = b->solve_ms;
    if (iterations) *iterations = b->iters_run;
    return 0;
}

}  // extern "C"
