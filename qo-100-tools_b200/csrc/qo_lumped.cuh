/*
 * qo_lumped.cuh -- the FP64-FMA-bound hot kernel (sm_100a).
 *
 * One warp owns one Monte-Carlo sample at a time; each lane owns that sample's
 * (sample, frequency) points two at a time (one double2 load = two adjacent grid
 * frequencies) and chains the complex 2x2 ABCD products of all elements in
 * registers.  Per sample the warp first derives the perturbed, hoisted element
 * coefficients (Philox -> value -> 1/C, L*Cp, ...) into a shared-memory table
 * that all lanes then read by broadcast.  |S21|^2 / |S11|^2 are compared against
 * the specs in linear power (no log in the loop); pass/fail and the histogram
 * variable are reduced with warp shuffles, then shared-memory atomics, then one
 * global atomic per counter per block.
 *
 * ABCD conventions (SURVEY App. B.1): series Z: B += A*Z, D += C*Z;
 * shunt Y: A += B*Y, C += D*Y; product runs source -> load.
 */
#pragma once
#include "qo_device.cuh"
#include "qo_stream.h"

#define QO_TPB 256
#define QO_WARPS (QO_TPB / 32)

/* ---- scalar helpers, generic over double / float ------------------------- */
__device__ __forceinline__ double qfma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float qfma(float a, float b, float c) { return fmaf(a, b, c); }

/* 1/x: MUFU.RCP64H seed (>= 20 good bits) + one cubic step: e = 1 - x*r0,
 * r = r0*(1 + e + e^2); relative error ~e^3 + 1 rounding (validated on device in
 * tests/test_gpu_parity.py::test_rcp_accuracy). 3 DFMA instead of the 4 of two
 * Newton steps, and no slow-path branch. */
__device__ __forceinline__ double qrcp(double x)
{
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(x));
    double e = fma(-x, r0, 1.0);
    double t = fma(e, e, e);
    return fma(r0, t, r0);
}
__device__ __forceinline__ float qrcp(float x) { return __frcp_rn(x); }

__device__ __forceinline__ void qsincos(double x, double *s, double *c) { sincos(x, s, c); }
__device__ __forceinline__ void qsincos(float x, float *s, float *c) { sincosf(x, s, c); }

template <typename T> struct QoVec2;
template <> struct QoVec2<double> { typedef double2 type; };
template <> struct QoVec2<float> { typedef float2 type; };

/* two (sample, frequency) points per thread */
template <typename T> struct Abcd2 {
    T ar[2], ai[2], br[2], bi[2], cr[2], ci[2], dr[2], di[2];
};

#define QO_P2 _Pragma("unroll") for (int p = 0; p < 2; p++)

/* ROW (run-time compiled flavour, jobs that observe |S21| only): the chain carries the row vector [1 Rs] M in (a, b) instead
 * of the 2x2 product -- den = a Rl + b -- and the (c, d) row is never touched: half the multiply-adds per element */
template <typename T, bool ROW = false> __device__ __forceinline__ void ser_cplx(Abcd2<T> &m, int p, T zr, T zi)
{
    m.br[p] = qfma(m.ar[p], zr, m.br[p]); m.br[p] = qfma(-m.ai[p], zi, m.br[p]);
    m.bi[p] = qfma(m.ar[p], zi, m.bi[p]); m.bi[p] = qfma(m.ai[p], zr, m.bi[p]);
    if (ROW) return;
    m.dr[p] = qfma(m.cr[p], zr, m.dr[p]); m.dr[p] = qfma(-m.ci[p], zi, m.dr[p]);
    m.di[p] = qfma(m.cr[p], zi, m.di[p]); m.di[p] = qfma(m.ci[p], zr, m.di[p]);
}
template <typename T, bool ROW = false> __device__ __forceinline__ void shunt_cplx(Abcd2<T> &m, int p, T yr, T yi)
{
    m.ar[p] = qfma(m.br[p], yr, m.ar[p]); m.ar[p] = qfma(-m.bi[p], yi, m.ar[p]);
    m.ai[p] = qfma(m.br[p], yi, m.ai[p]); m.ai[p] = qfma(m.bi[p], yr, m.ai[p]);
    if (ROW) return;
    m.cr[p] = qfma(m.dr[p], yr, m.cr[p]); m.cr[p] = qfma(-m.di[p], yi, m.cr[p]);
    m.ci[p] = qfma(m.dr[p], yi, m.ci[p]); m.ci[p] = qfma(m.di[p], yr, m.ci[p]);
}
template <typename T, bool ROW = false> __device__ __forceinline__ void ser_imag(Abcd2<T> &m, int p, T x)
{
    m.br[p] = qfma(-m.ai[p], x, m.br[p]); m.bi[p] = qfma(m.ar[p], x, m.bi[p]);
    if (ROW) return;
    m.dr[p] = qfma(-m.ci[p], x, m.dr[p]); m.di[p] = qfma(m.cr[p], x, m.di[p]);
}
template <typename T, bool ROW = false> __device__ __forceinline__ void shunt_imag(Abcd2<T> &m, int p, T y)
{
    m.ar[p] = qfma(-m.bi[p], y, m.ar[p]); m.ai[p] = qfma(m.br[p], y, m.ai[p]);
    if (ROW) return;
    m.cr[p] = qfma(-m.di[p], y, m.cr[p]); m.ci[p] = qfma(m.dr[p], y, m.ci[p]);
}
/* M <- M * [a b; c d] with a general complex 2x2 (TLINE / coupled line blocks) */
template <typename T, bool ROW = false>
__device__ __forceinline__ void mul_full(Abcd2<T> &m, int p, T ar, T ai, T br, T bi, T cr, T ci, T dr, T di)
{
    T Ar = m.ar[p], Ai = m.ai[p], Br = m.br[p], Bi = m.bi[p];
    m.ar[p] = qfma(Ar, ar, qfma(-Ai, ai, qfma(Br, cr, -Bi * ci)));
    m.ai[p] = qfma(Ar, ai, qfma(Ai, ar, qfma(Br, ci, Bi * cr)));
    m.br[p] = qfma(Ar, br, qfma(-Ai, bi, qfma(Br, dr, -Bi * di)));
    m.bi[p] = qfma(Ar, bi, qfma(Ai, br, qfma(Br, di, Bi * dr)));
    if (ROW) return;
    T Cr = m.cr[p], Ci = m.ci[p], Dr = m.dr[p], Di = m.di[p];
    m.cr[p] = qfma(Cr, ar, qfma(-Ci, ai, qfma(Dr, cr, -Di * ci)));
    m.ci[p] = qfma(Cr, ai, qfma(Ci, ar, qfma(Dr, ci, Di * cr)));
    m.dr[p] = qfma(Cr, br, qfma(-Ci, bi, qfma(Dr, dr, -Di * di)));
    m.di[p] = qfma(Cr, bi, qfma(Ci, br, qfma(Dr, di, Di * dr)));
}

/* ---- the element chain for two points ------------------------------------ */
struct QoPlanes {
    double2 *s11, *s21, *s12, *s22;
    /* measured two-port blocks (OP_SBLOCK): ABCD per (block, grid point) as four double2, and the product of the
     * blocks' determinants per grid point (NULL when every block is reciprocal) */
    const double2 *sblk, *sdet;
    int npts;
    const double *cplms;        /* physical coupled-line element: per-sample Z0e, Z0o, theta_e, theta_o from the pre-pass */
};

#ifdef QO_JIT_CHAIN
#define QO_ROW QO_JIT_ROW
#else
#define QO_ROW false
#endif
/* one element: M <- M * ABCD(op; cf) at the two points.  The interpreter calls it with the opcode read from shared memory;
 * the run-time compiled flavour (qo_chain_jit.h) calls it once per element with literal arguments, so that the switch folds away */
template <typename T, bool TRIG, bool ROW = false>
__device__ __forceinline__ void qo_chain_step(const int op, const T *__restrict__ cf, const T (&w)[2], const T (&wi)[2],
                                              const T (&w2)[2], Abcd2<T> &m, const QoPlanes &planes, int k0)
{
    {
        switch (op) {
        case OP_SER_LOSSY_L: {   /* Z = (R + jwL) / (1 - w^2 L Cp + j w R Cp) */
            T L = cf[0], LCp = cf[1], R = cf[2], RCp = cf[3];
            QO_P2 {
                T dre = qfma(-w2[p], LCp, T(1)), dim = w[p] * RCp, xl = w[p] * L;
                T r = qrcp(qfma(dre, dre, dim * dim));
                T qr = dre * r, qi = -dim * r;
                ser_cplx<T, ROW>(m, p, qfma(R, qr, -xl * qi), qfma(R, qi, xl * qr));
            }
            break;
        }
        case OP_SHUNT_LOSSY_C: {  /* Y = 1 / (R + j(w Ls - 1/(wC))) */
            T Ci = cf[0], Ls = cf[1], R = cf[2], R2 = cf[3];
            QO_P2 {
                T x = qfma(w[p], Ls, -wi[p] * Ci);
                T r = qrcp(qfma(x, x, R2));
                shunt_cplx<T, ROW>(m, p, R * r, -x * r);
            }
            break;
        }
        case OP_SER_LOSSY_C: {
            T Ci = cf[0], Ls = cf[1], R = cf[2];
            QO_P2 ser_cplx<T, ROW>(m, p, R, qfma(w[p], Ls, -wi[p] * Ci));
            break;
        }
        case OP_SHUNT_LOSSY_L: {  /* Y = (1 - w^2 L Cp + j w R Cp) / (R + jwL) */
            T L = cf[0], LCp = cf[1], R = cf[2], RCp = cf[3];
            QO_P2 {
                T dre = qfma(-w2[p], LCp, T(1)), dim = w[p] * RCp, xl = w[p] * L;
                T r = qrcp(qfma(xl, xl, R * R));
                T qr = R * r, qi = -xl * r;
                shunt_cplx<T, ROW>(m, p, qfma(dre, qr, -dim * qi), qfma(dre, qi, dim * qr));
            }
            break;
        }
        case OP_SER_R: { T r = cf[0]; QO_P2 {
            m.br[p] = qfma(m.ar[p], r, m.br[p]); m.bi[p] = qfma(m.ai[p], r, m.bi[p]);
            if (!ROW) { m.dr[p] = qfma(m.cr[p], r, m.dr[p]); m.di[p] = qfma(m.ci[p], r, m.di[p]); } } break; }
        case OP_SHUNT_G: { T g = cf[0]; QO_P2 {
            m.ar[p] = qfma(m.br[p], g, m.ar[p]); m.ai[p] = qfma(m.bi[p], g, m.ai[p]);
            if (!ROW) { m.cr[p] = qfma(m.dr[p], g, m.cr[p]); m.ci[p] = qfma(m.di[p], g, m.ci[p]); } } break; }
        case OP_SER_L: { T c0 = cf[0]; QO_P2 ser_imag<T, ROW>(m, p, w[p] * c0); break; }
        case OP_SER_C: { T c0 = cf[0]; QO_P2 ser_imag<T, ROW>(m, p, -wi[p] * c0); break; }
        case OP_SER_LCS: { T c0 = cf[0], c1 = cf[1]; QO_P2 ser_imag<T, ROW>(m, p, qfma(w[p], c0, -wi[p] * c1)); break; }
        case OP_SHUNT_C: { T c0 = cf[0]; QO_P2 shunt_imag<T, ROW>(m, p, w[p] * c0); break; }
        case OP_SHUNT_L: { T c0 = cf[0]; QO_P2 shunt_imag<T, ROW>(m, p, -wi[p] * c0); break; }
        case OP_SHUNT_LCP: { T c0 = cf[0], c1 = cf[1]; QO_P2 shunt_imag<T, ROW>(m, p, qfma(w[p], c0, -wi[p] * c1)); break; }
        case OP_SER_LCP: { T c0 = cf[0], c1 = cf[1]; QO_P2 ser_imag<T, ROW>(m, p, -qrcp(qfma(w[p], c0, -wi[p] * c1))); break; }
        case OP_SHUNT_LCS: { T c0 = cf[0], c1 = cf[1]; QO_P2 shunt_imag<T, ROW>(m, p, -qrcp(qfma(w[p], c0, -wi[p] * c1))); break; }
        default:
            if (TRIG) {
                if (op == OP_TLINE) {
                    T z0 = cf[0], y0 = cf[1], kt = cf[2];
                    QO_P2 {
                        T s, c;
                        qsincos(kt * w[p], &s, &c);
                        mul_full<T, ROW>(m, p, c, T(0), T(0), z0 * s, T(0), s * y0, c, T(0));
                    }
                } else if (op == OP_CPL) {
                    /* even/odd-mode lines in a Zt system (SURVEY B.4) */
                    T cE = cf[0], dE = cf[1], cO = cf[2], dO = cf[3], ke = cf[4], ko = cf[5], zt = cf[6], yt = cf[7];
                    QO_P2 {
                        T se, ce, so, co;
                        qsincos(ke * w[p], &se, &ce);
                        qsincos(ko * w[p], &so, &co);
                        /* 1/den_e, 1/den_o ; den = 2c + j s cX */
                        T er_ = ce + ce, ei_ = se * cE, or_ = co + co, oi_ = so * cO;
                        T re = qrcp(qfma(er_, er_, ei_ * ei_)), ro = qrcp(qfma(or_, or_, oi_ * oi_));
                        T ier = er_ * re, iei = -ei_ * re, ior = or_ * ro, ioi = -oi_ * ro;
                        /* s21 = (Te+To)/2 = ie + io ; s11 = (j se dE ie + j so dO io)/2 */
                        T s21r = ier + ior, s21i = iei + ioi;
                        T ge = T(0.5) * se * dE, go = T(0.5) * so * dO;
                        T s11r = -(ge * iei + go * ioi), s11i = ge * ier + go * ior;
                        /* symmetric S -> ABCD at Zt */
                        T q2r = s21r * s21r - s21i * s21i, q2i = T(2) * s21r * s21i;      /* s21^2 */
                        T p2r = s11r * s11r - s11i * s11i, p2i = T(2) * s11r * s11i;      /* s11^2 */
                        T dr_ = s21r + s21r, di_ = s21i + s21i;
                        T rd = qrcp(qfma(dr_, dr_, di_ * di_));
                        T idr = dr_ * rd, idi = -di_ * rd;                                /* 1/(2 s21) */
                        T nar = T(1) - p2r + q2r, nai = q2i - p2i;                        /* 1 - s11^2 + s21^2 */
                        T nbr = T(1) + s11r + s11r + p2r - q2r, nbi = s11i + s11i + p2i - q2i; /* (1+s11)^2 - s21^2 */
                        T ncr = T(1) - s11r - s11r + p2r - q2r, nci = -s11i - s11i + p2i - q2i;
                        T Ar = nar * idr - nai * idi, Ai = nar * idi + nai * idr;
                        T Br = zt * (nbr * idr - nbi * idi), Bi = zt * (nbr * idi + nbi * idr);
                        T Cr = yt * (ncr * idr - nci * idi), Ci2 = yt * (ncr * idi + nci * idr);
                        mul_full<T, ROW>(m, p, Ar, Ai, Br, Bi, Cr, Ci2, Ar, Ai);
                    }
                } else if (op == OP_SBLOCK) {
                    const int blk = (int)cf[0];
                    QO_P2 {
                        const int k = min(k0 + p, planes.npts - 1);
                        const double2 *t = planes.sblk + ((size_t)blk * (size_t)planes.npts + (size_t)k) * 4;
                        const double2 a = t[0], b = t[1], c = t[2], d = t[3];
                        mul_full<T, ROW>(m, p, T(a.x), T(a.y), T(b.x), T(b.y), T(c.x), T(c.y), T(d.x), T(d.y));
                    }
                }
            }
            break;
        }
    }
}

template <typename T, bool TRIG>
__device__ __forceinline__ void qo_chain2(const int *__restrict__ s_op, const int *__restrict__ s_coff,
                                          const T *__restrict__ coef, int n_ops, const T (&w)[2], const T (&wi)[2],
                                          Abcd2<T> &m, const QoPlanes &planes, int k0)
{
    if (!QO_ROW) {               /* QO_ROW: the caller has put [1 Rs] into (a, b) */
        QO_P2 { m.ar[p] = T(1); m.ai[p] = T(0); m.br[p] = T(0); m.bi[p] = T(0);
                m.cr[p] = T(0); m.ci[p] = T(0); m.dr[p] = T(1); m.di[p] = T(0); }
    }
    T w2[2];
    QO_P2 w2[p] = w[p] * w[p];
#ifdef QO_JIT_CHAIN
    QO_JIT_CHAIN                 /* qo_chain_step<T, TRIG, QO_ROW>(<opcode>, coef + <offset>, w, wi, w2, m, planes, k0); per element */
#else
    for (int e = 0; e < n_ops; e++) qo_chain_step<T, TRIG>(s_op[e], coef + s_coff[e], w, wi, w2, m, planes, k0);
#endif
}

/* ---- per-sample coefficient derivation (one lane per element) ------------- */
template <typename T>
__device__ __forceinline__ void qo_derive(const DevProg *__restrict__ prog, int e, const double *__restrict__ x, T *out,
                                          const double *__restrict__ cplms)
{
    double p[6];
#pragma unroll
    for (int k = 0; k < 6; k++) {
        p[k] = prog->nom[e][k];
        int tv = prog->tvar[e][k];
        if (tv >= 0) p[k] = qo_stream_apply(p[k], prog->ttol[e][k], x[tv], prog->tmode[e][k]);
    }
    if (e == prog->cplms_elem) {
        /* physical coupled line: p[] holds (W, S, L, H_t, f0, Zt); the electrical view of THIS sample was computed by
         * the pre-pass from the same draws */
        p[0] = cplms[0]; p[1] = cplms[1]; p[2] = cplms[2]; p[3] = cplms[3]; p[4] = prog->nom[e][4]; p[5] = prog->nom[e][5];
    }
    switch (prog->opcode[e]) {
    case OP_SER_R: out[0] = T(p[0]); break;
    case OP_SHUNT_G: out[0] = T(1.0 / p[0]); break;
    case OP_SER_L: out[0] = T(p[0]); break;
    case OP_SER_C: out[0] = T(1.0 / p[0]); break;
    case OP_SHUNT_C: out[0] = T(p[0]); break;
    case OP_SHUNT_L: out[0] = T(1.0 / p[0]); break;
    case OP_SER_LCS: case OP_SHUNT_LCS: out[0] = T(p[0]); out[1] = T(1.0 / p[1]); break;   /* (L, 1/C) */
    case OP_SER_LCP: case OP_SHUNT_LCP: out[0] = T(p[1]); out[1] = T(1.0 / p[0]); break;   /* (C, 1/L) */
    case OP_SER_LOSSY_L: case OP_SHUNT_LOSSY_L:
        out[0] = T(p[0]); out[1] = T(p[0] * p[2]); out[2] = T(p[1]); out[3] = T(p[1] * p[2]); break;
    case OP_SER_LOSSY_C: case OP_SHUNT_LOSSY_C:
        out[0] = T(1.0 / p[0]); out[1] = T(p[2]); out[2] = T(p[1]); out[3] = T(p[1] * p[1]); break;
    case OP_TLINE: out[0] = T(p[0]); out[1] = T(1.0 / p[0]); out[2] = T(p[1] / (360.0 * p[2])); break;
    case OP_SBLOCK: out[0] = T(p[0]); break;
    case OP_CPL: {
        double a = p[0] / p[5], b = p[1] / p[5];
        out[0] = T(a + 1.0 / a); out[1] = T(a - 1.0 / a); out[2] = T(b + 1.0 / b); out[3] = T(b - 1.0 / b);
        out[4] = T(p[2] / (360.0 * p[4])); out[5] = T(p[3] / (360.0 * p[4])); out[6] = T(p[5]); out[7] = T(1.0 / p[5]);
        break;
    }
    default: break;
    }
}

/* 32 contiguous bytes (two complex doubles) in one 256-bit store; p must be 32-byte aligned */
__device__ __forceinline__ void qo_st256(double2 *p, double2 a, double2 b)
{
#ifdef QO_NO_ST256          /* run-time compilation by an NVRTC older than CUDA 12.9 (qo_chain_jit.h) */
    p[0] = a; p[1] = b;
#else
    asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" :: "l"(p), "d"(a.x), "d"(a.y), "d"(b.x), "d"(b.y) : "memory");
#endif
}

/* ---- the kernel ----------------------------------------------------------- */
/* Compiled ahead of time this is the opcode interpreter.  qo_chain_jit.h hands the same text to NVRTC with the job's element
 * list (QO_JIT_CHAIN), spec kinds and template arguments defined in front of it: one kernel, C linkage, no dispatch. */
#ifdef QO_JIT_CHAIN
extern "C" __global__ void __launch_bounds__(QO_TPB, 2)
qo_mc_chain_jit_kernel(
#else
//@mu{ MU: the stability spec (SK_MU_MIN) on the full 2x2 product; the chain kernel of every other job keeps the head below
template <typename T, bool FULL_S, bool TRIG, bool GD, bool S22, bool MU>
#if 0
//@mu}
template <typename T, bool FULL_S, bool TRIG, bool GD, bool S22>
//@mu{
#endif
//@mu}
__global__ void __launch_bounds__(QO_TPB, 2)
qo_mc_lumped_kernel(
#endif
                    const DevProg *__restrict__ prog, const typename QoVec2<T>::type *__restrict__ w2,
                    const typename QoVec2<T>::type *__restrict__ wi2, const uchar2 *__restrict__ m2, int nf, int npairs,
                    int pairs_per_chunk, int nchunks, unsigned long long sample_offset, unsigned long long nsamples,
                    unsigned long long *__restrict__ counters, QoPlanes planes)
{
    __shared__ int s_op[QO_MAX_OPS], s_coff[QO_MAX_OPS];
    __shared__ __align__(16) T s_coef[QO_WARPS][QO_MAX_COEF];
    __shared__ double s_x[QO_WARPS][QO_MAX_VAR];
    __shared__ unsigned int s_cnt[QO_NCNT_MAX];
    __shared__ T s_thr[QO_NSPEC_MAX];
    __shared__ int s_sk[QO_NSPEC_MAX];
    __shared__ double s_gdthr[QO_NSPEC_MAX];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#ifdef QO_JIT_CHAIN
    constexpr int n_ops = QO_JIT_NOPS, nspec = QO_JIT_NSPEC, hist_spec = QO_JIT_HIST_SPEC, hist_kind = QO_JIT_HIST_KIND;
    constexpr bool need_s11 = FULL_S || QO_JIT_NEED_S11;
    const int n_var = prog->n_var;
#define QO_SK(sp) qj_sk(sp)
#else
    const int n_ops = prog->n_ops, n_var = prog->n_var, nspec = prog->nspec;
    const int hist_spec = prog->hist_bins > 0 ? prog->hist_spec : -1;
    const bool need_s11 = FULL_S || prog->need_s11;
#define QO_SK(sp) s_sk[sp]
#endif
    const int ncnt = qo_ncnt(nspec, prog->hist_bins);
    const bool planes_al32 = ((((size_t)planes.s11) | ((size_t)planes.s21) | ((size_t)planes.s12) | ((size_t)planes.s22)) & 31) == 0;
    for (int i = threadIdx.x; i < n_ops; i += QO_TPB) { s_op[i] = prog->opcode[i]; s_coff[i] = prog->coff[i]; }
    qo_tally_zero<QO_TPB>(s_cnt, ncnt);
    if (threadIdx.x < QO_NSPEC_MAX) {
        s_thr[threadIdx.x] = T(prog->spec_thr[threadIdx.x]); s_sk[threadIdx.x] = prog->spec_kind[threadIdx.x];
        s_gdthr[threadIdx.x] = prog->spec_thr[threadIdx.x];
    }
    const unsigned int gd_bits = GD ? (unsigned int)prog->need_gd : 0u;     /* bit sp set: spec sp is a group-delay spec */
    __syncthreads();

    const T rs = T(prog->rs), rl = T(prog->rl), rsrl = T(prog->rsrl), k21 = T(prog->k21);
#ifndef QO_JIT_CHAIN
    const int hist_kind = hist_spec >= 0 ? prog->spec_kind[hist_spec] : 0;
#endif
    const unsigned long long seed = prog->seed;
    const int dist = prog->dist;
    T *coefw = s_coef[warp];
    double *xw = s_x[warp];

    const unsigned long long total_warps = (unsigned long long)gridDim.x * QO_WARPS;
    const unsigned long long n_units = nsamples * (unsigned long long)nchunks;
    for (unsigned long long u = (unsigned long long)blockIdx.x * QO_WARPS + warp; u < n_units; u += total_warps) {
        const unsigned long long s = nchunks == 1 ? u : u / (unsigned long long)nchunks;
        const int chunk = nchunks == 1 ? 0 : (int)(u - s * (unsigned long long)nchunks);
        /* 1. this sample's random variables, one lane each (Philox is counter-based: no state) */
        for (int v = lane; v < n_var; v += 32) xw[v] = qo_stream_variate(seed, sample_offset + s, (uint32_t)v, dist);
        __syncwarp();
        /* 2. perturbed + hoisted element coefficients -> shared table */
        for (int e = lane; e < n_ops; e += 32) qo_derive<T>(prog, e, xw, coefw + s_coff[e], planes.cplms ? planes.cplms + 4 * s : NULL);
        __syncwarp();

        /* 3. frequency loop: two points per lane per iteration */
        unsigned int fail = 0;
        T wn = T(0), wd = T(1);
//@mu{
        if (MU && hist_kind == SK_MU_MIN) { wn = T(-1); wd = T(0); }    /* -mu = -infinity: the first in-band point replaces it */
//@mu}
        double gd_worst = -1e300;        /* largest group delay seen in the histogram spec's band (GD specs) */
        const int lo = chunk * pairs_per_chunk;
        const int hi = min(npairs, lo + pairs_per_chunk);
        int j = lo + lane;
        typename QoVec2<T>::type wv, wiv;
        uchar2 mv = make_uchar2(0, 0);
        if (j < hi) { wv = w2[j]; wiv = wi2[j]; if (!FULL_S) mv = m2[j]; }
        while (j < hi) {
            const T w[2] = { wv.x, wv.y }, wi[2] = { wiv.x, wiv.y };
            const unsigned int mk[2] = { mv.x, mv.y };
            const int jn = j + 32;
            if (jn < hi) { wv = w2[jn]; wiv = wi2[jn]; if (!FULL_S) mv = m2[jn]; }   /* prefetch next pair */
            Abcd2<T> m;
            if (QO_ROW) { QO_P2 { m.ar[p] = T(1); m.ai[p] = T(0); m.br[p] = rs; m.bi[p] = T(0); } }
            qo_chain2<T, TRIG>(s_op, s_coff, coefw, n_ops, w, wi, m, planes, 2 * j);
            double2 o11[2], o21[2], o22[2];
            QO_P2 {
                /* den = A Rl + B + C Rs Rl + D Rs ; n11 = A Rl + B - C Rs Rl - D Rs */
                T den_r, den_i, n_r = T(0), n_i = T(0), num2 = T(0), num22 = T(0);
                if (need_s11) {
                    T pr = qfma(m.ar[p], rl, m.br[p]), pi_ = qfma(m.ai[p], rl, m.bi[p]);
                    T qr = qfma(m.cr[p], rsrl, m.dr[p] * rs), qi = qfma(m.ci[p], rsrl, m.di[p] * rs);
                    den_r = pr + qr; den_i = pi_ + qi; n_r = pr - qr; n_i = pi_ - qi;
                    num2 = qfma(n_r, n_r, n_i * n_i);
                } else if (QO_ROW) {
                    den_r = qfma(m.ar[p], rl, m.br[p]); den_i = qfma(m.ai[p], rl, m.bi[p]);
                } else {
                    den_r = qfma(m.dr[p], rs, qfma(m.cr[p], rsrl, qfma(m.ar[p], rl, m.br[p])));
                    den_i = qfma(m.di[p], rs, qfma(m.ci[p], rsrl, qfma(m.ai[p], rl, m.bi[p])));
                }
                const T den2 = qfma(den_r, den_r, den_i * den_i);
                if (S22 && !FULL_S) {
                    /* n22 = -A Rl + B - C Rs Rl + D Rs; on the row vector (a, b) = [1 Rs] M that is -a Rl + b */
                    T xr, xi;
                    if (QO_ROW) { xr = qfma(-m.ar[p], rl, m.br[p]); xi = qfma(-m.ai[p], rl, m.bi[p]); }
                    else {
                        xr = qfma(-m.ar[p], rl, m.br[p]) + qfma(-m.cr[p], rsrl, m.dr[p] * rs);
                        xi = qfma(-m.ai[p], rl, m.bi[p]) + qfma(-m.ci[p], rsrl, m.di[p] * rs);
                    }
                    num22 = qfma(xr, xr, xi * xi);
                }
//@mu{
                /* Edwards-Sinsky mu = (1 - |S11|^2) / (|S22 - Delta conj(S11)| + |S12 S21|), Delta = S11 S22 - S12 S21, with
                 * S11 = n11/D, S22 = n22/D, S21 = k21/D, S12 = k21 det/D (det: the blocks' product of AD - BC, 1 when every block
                 * is reciprocal).  Multiplied through by |D|^3: mu = mu_n / mu_d, mu_n = (|D|^2 - |n11|^2) |D|,
                 * mu_d = |X| + k21^2 |det| |D|, X = n22 (|D|^2 - |n11|^2) + k21^2 det conj(n11).  mu_d >= 0, so the verdict
                 * needs no division and the worst-value tracker below orders -mu = -mu_n / mu_d correctly though mu may be < 0. */
                T mu_n = T(0), mu_d = T(1);
                if (MU && !FULL_S) {
                    const T ur = qfma(-m.ar[p], rl, m.br[p]) + qfma(-m.cr[p], rsrl, m.dr[p] * rs);
                    const T ui = qfma(-m.ai[p], rl, m.bi[p]) + qfma(-m.ci[p], rsrl, m.di[p] * rs);
                    T dtr = T(1), dti = T(0);
                    if (planes.sdet) { const double2 dt = planes.sdet[min(2 * j + p, planes.npts - 1)]; dtr = T(dt.x); dti = T(dt.y); }
                    const T g = den2 - num2, kk = k21 * k21, aden = sqrt(den2);
                    const T xr = qfma(ur, g, kk * qfma(dtr, n_r, dti * n_i)), xi = qfma(ui, g, kk * qfma(dti, n_r, -dtr * n_i));
                    mu_n = g * aden;
                    mu_d = qfma(kk * sqrt(qfma(dtr, dtr, dti * dti)), aden, sqrt(qfma(xr, xr, xi * xi)));
                }
//@mu}
                if (FULL_S) {
                    const T r = qrcp(den2);
                    const T ir = den_r * r, ii = -den_i * r;
                    o21[p] = make_double2((double)(k21 * ir), (double)(k21 * ii));
                    o11[p] = make_double2((double)(n_r * ir - n_i * ii), (double)(n_r * ii + n_i * ir));
                    /* n22 = -A Rl + B - C Rs Rl + D Rs */
                    T ur = qfma(-m.ar[p], rl, m.br[p]), ui = qfma(-m.ai[p], rl, m.bi[p]);
                    T vr = qfma(-m.cr[p], rsrl, m.dr[p] * rs), vi = qfma(-m.ci[p], rsrl, m.di[p] * rs);
                    T xr = ur + vr, xi = ui + vi;
                    o22[p] = make_double2((double)(xr * ir - xi * ii), (double)(xr * ii + xi * ir));
                } else {
                    const unsigned int mb = mk[p];
                    double gdv = 0.0;
                    if (GD && (gd_bits & mb)) {
                        /* group delay tau = -d(arg S21)/dw by the central difference the sweep API and the oracle use:
                         * the chain is re-evaluated at w (1 +- 1e-6); arg S21 = -arg den.  Only points inside a
                         * GD spec band pay for it. */
                        const T dwq = w[p] * T(1e-6);
                        const T wq[2] = { w[p] + dwq, w[p] - dwq };
                        const T wiq[2] = { T(1) / wq[0], T(1) / wq[1] };
                        Abcd2<T> mg;
                        if (QO_ROW) { _Pragma("unroll") for (int q = 0; q < 2; q++) { mg.ar[q] = T(1); mg.ai[q] = T(0); mg.br[q] = rs; mg.bi[q] = T(0); } }
                        qo_chain2<T, TRIG>(s_op, s_coff, coefw, n_ops, wq, wiq, mg, planes, 2 * j);
                        T dgr[2], dgi[2];
#pragma unroll
                        for (int q = 0; q < 2; q++) {
                            if (QO_ROW) { dgr[q] = qfma(mg.ar[q], rl, mg.br[q]); dgi[q] = qfma(mg.ai[q], rl, mg.bi[q]); continue; }
                            dgr[q] = qfma(mg.dr[q], rs, qfma(mg.cr[q], rsrl, qfma(mg.ar[q], rl, mg.br[q])));
                            dgi[q] = qfma(mg.di[q], rs, qfma(mg.ci[q], rsrl, qfma(mg.ai[q], rl, mg.bi[q])));
                        }
                        const double cre = (double)dgr[0] * (double)dgr[1] + (double)dgi[0] * (double)dgi[1];
                        const double cim = (double)dgi[0] * (double)dgr[1] - (double)dgr[0] * (double)dgi[1];
                        gdv = atan2(cim, cre) / (2.0 * (double)dwq);
                    }
#pragma unroll
                    for (int sp = 0; sp < QO_NSPEC_MAX; sp++) {
                        if (sp < nspec) {
                            const int sk = QO_SK(sp);
                            const T thr = s_thr[sp];
                            bool bad = sk == SK_DEN2_MAX ? (den2 > thr) : sk == SK_DEN2_MIN ? (den2 < thr)
                                     : sk == SK_S11_MAX ? (num2 > thr * den2) : (S22 && sk == SK_S22_MAX) ? (num22 > thr * den2)
                                     : (gdv > s_gdthr[sp]);
//@mu{
                            if (MU && sk == SK_MU_MIN) bad = !(mu_n >= thr * mu_d);     /* !(mu >= limit): NaN fails */
//@mu}
                            if (bad && ((mb >> sp) & 1u)) fail |= 1u << sp;
                        }
                    }
                    if (GD && hist_kind == SK_GD_MAX && hist_spec >= 0 && ((mb >> hist_spec) & 1u) && gdv > gd_worst) gd_worst = gdv;
                    if (hist_spec >= 0 && hist_kind != SK_GD_MAX && ((mb >> hist_spec) & 1u)) {
                        /* track the worst value as a ratio a/b ("larger is worse") without dividing */
                        T a = hist_kind == SK_DEN2_MAX ? den2 : hist_kind == SK_DEN2_MIN ? T(1) : (S22 && hist_kind == SK_S22_MAX) ? num22 : num2;
                        T b = hist_kind == SK_DEN2_MAX ? T(1) : den2;
//@mu{
                        if (MU && hist_kind == SK_MU_MIN) { a = -mu_n; b = mu_d; }
//@mu}
                        if (a * wd > wn * b) { wn = a; wd = b; }
                    }
                }
            }
            if (FULL_S) {
                /* A lane owns two ADJACENT points = 32 contiguous bytes per plane: one 256-bit store per plane
                 * (STG.E.ENL2.256) makes every warp store a full 1 KB run.  Two 16-byte stores per lane leave
                 * every 32-byte sector half written per instruction (ncu r01d: 16 of 32 bytes per sector used,
                 * DRAM at 41 % of peak).  S12 = S21 (AD - BC) with AD - BC == 1 exactly: every element is
                 * reciprocal, and the numerical determinant cancels catastrophically in a deep stop band. */
                const int k = 2 * j;
                const size_t o = (size_t)s * (size_t)nf + (size_t)k;
                double2 o12[2] = { o21[0], o21[1] };
                if (TRIG && planes.sdet) {       /* non-reciprocal measured blocks: S12 = S21 * prod det(block) */
                    QO_P2 {
                        const double2 dt = planes.sdet[min(k + p, planes.npts - 1)];
                        o12[p] = make_double2(o21[p].x * dt.x - o21[p].y * dt.y, o21[p].x * dt.y + o21[p].y * dt.x);
                    }
                }
                if (k + 1 < nf && ((o & 1) == 0) && planes_al32) {
                    if (planes.s21) qo_st256(planes.s21 + o, o21[0], o21[1]);
                    if (planes.s11) qo_st256(planes.s11 + o, o11[0], o11[1]);
                    if (planes.s22) qo_st256(planes.s22 + o, o22[0], o22[1]);
                    if (planes.s12) qo_st256(planes.s12 + o, o12[0], o12[1]);
                } else {
                    QO_P2 {
                        if (k + p < nf) {
                            if (planes.s21) planes.s21[o + p] = o21[p];
                            if (planes.s11) planes.s11[o + p] = o11[p];
                            if (planes.s22) planes.s22[o + p] = o22[p];
                            if (planes.s12) planes.s12[o + p] = o12[p];
                        }
                    }
                }
            }
            j = jn;
        }

        if (!FULL_S) {
            /* 4. warp-shuffle reduction, then block-level shared atomics */
            fail = __reduce_or_sync(0xffffffffu, fail);
            if (hist_spec >= 0) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    T on = __shfl_xor_sync(0xffffffffu, wn, off), od = __shfl_xor_sync(0xffffffffu, wd, off);
                    if (on * wd > wn * od) { wn = on; wd = od; }
                    if (GD) {
                        const double og = __shfl_xor_sync(0xffffffffu, gd_worst, off);
                        if (og > gd_worst) gd_worst = og;
                    }
                }
            }
            if (lane == 0) {
                qo_tally_one(s_cnt, nspec, fail);
                if (hist_spec >= 0) {
                    double ratio = (double)wn / (double)wd;
                    double lin = hist_kind == SK_S11_MAX || (S22 && hist_kind == SK_S22_MAX) ? ratio
                               : hist_kind == SK_DEN2_MAX ? (double)k21 * (double)k21 / ratio
                                                          : (double)k21 * (double)k21 * ratio;
                    double v = hist_kind == SK_GD_MAX ? gd_worst : 10.0 * log10(lin);
//@mu{
                    if (MU && hist_kind == SK_MU_MIN) v = -ratio;               /* the in-band minimum of mu, linear */
//@mu}
                    qo_tally_hist(s_cnt, nspec, qo_hist_bin(v, prog->hist_lo, prog->hist_hi, prog->hist_bins));
                }
            }
        }
        __syncwarp();
    }
    if (!FULL_S) {
        __syncthreads();
        qo_tally_flush<QO_TPB>(s_cnt, ncnt, counters);
    }
}
#undef QO_SK
#undef QO_ROW
