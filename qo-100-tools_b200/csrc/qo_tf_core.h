/*
 * qo_tf_core.h -- element -> rational immittance, shared by the transfer-function kernel (qo_tf.cuh, device) and
 * its plan-time self-check (qo_tf.cu, host).
 *
 * Every lumped branch of the util/ networks (reference: util/if-bandpass-filter/schematic.svg:191-213 series-LC /
 * parallel-LC branches, util/gpsdo-ouput-filters/10M/schematic.svg:197-231, docs/gpsdo-filters/<name>.svg:195-241 traps,
 * pcb/generic-filter/qo-100-generic-filter.sch:1450-1488 ladder positions with the ESR/SRF parasitic model of
 * SURVEY 8d) has an immittance that is a ratio of real polynomials of degree <= 2 in s = jw:
 *     series branch  Z(s) = N(s) / D(s)          shunt branch  Y(s) = N(s) / D(s)
 * With sn = s / wref (wref = geometric centre of the grid) the coefficient of sn^k carries wref^k.
 */
#pragma once
#include "qo_device.cuh"

#if defined(__CUDACC__)
#define QO_TF_HD __host__ __device__ __forceinline__
#else
#define QO_TF_HD static inline
#endif

/* p[] = the element's (perturbed) parameters in the order of include/qo100net.h; nd[0..2] = N, nd[3..5] = D.
 * returns 1 for a series branch, 0 for a shunt branch, -1 when the opcode has no lumped rational form */
QO_TF_HD int qo_tf_element(int opcode, const double *p, double wr, double *nd)
{
    const double wr2 = wr * wr;
    switch (opcode) {
    case OP_SER_R: nd[0] = p[0]; nd[1] = 0; nd[2] = 0; nd[3] = 1; nd[4] = 0; nd[5] = 0; return 1;
    case OP_SHUNT_G: nd[0] = 1; nd[1] = 0; nd[2] = 0; nd[3] = p[0]; nd[4] = 0; nd[5] = 0; return 0;
    /* inductor (L, R, Cp): Z = (R + sL) / (1 + s R Cp + s^2 L Cp) */
    case OP_SER_L: case OP_SER_LOSSY_L:
        nd[0] = p[1]; nd[1] = p[0] * wr; nd[2] = 0; nd[3] = 1; nd[4] = p[1] * p[2] * wr; nd[5] = p[0] * p[2] * wr2; return 1;
    case OP_SHUNT_L: case OP_SHUNT_LOSSY_L:
        nd[3] = p[1]; nd[4] = p[0] * wr; nd[5] = 0; nd[0] = 1; nd[1] = p[1] * p[2] * wr; nd[2] = p[0] * p[2] * wr2; return 0;
    /* capacitor (C, R, Ls): Z = (1 + s R C + s^2 Ls C) / (s C) */
    case OP_SER_C: case OP_SER_LOSSY_C:
        nd[0] = 1; nd[1] = p[1] * p[0] * wr; nd[2] = p[2] * p[0] * wr2; nd[3] = 0; nd[4] = p[0] * wr; nd[5] = 0; return 1;
    case OP_SHUNT_C: case OP_SHUNT_LOSSY_C:
        nd[3] = 1; nd[4] = p[1] * p[0] * wr; nd[5] = p[2] * p[0] * wr2; nd[0] = 0; nd[1] = p[0] * wr; nd[2] = 0; return 0;
    /* ideal LC pairs (L, C) */
    case OP_SER_LCS:   /* Z = sL + 1/(sC) */
        nd[0] = 1; nd[1] = 0; nd[2] = p[0] * p[1] * wr2; nd[3] = 0; nd[4] = p[1] * wr; nd[5] = 0; return 1;
    case OP_SER_LCP:   /* Z = sL / (1 + s^2 L C) */
        nd[0] = 0; nd[1] = p[0] * wr; nd[2] = 0; nd[3] = 1; nd[4] = 0; nd[5] = p[0] * p[1] * wr2; return 1;
    case OP_SHUNT_LCS: /* Y = sC / (1 + s^2 L C) */
        nd[0] = 0; nd[1] = p[1] * wr; nd[2] = 0; nd[3] = 1; nd[4] = 0; nd[5] = p[0] * p[1] * wr2; return 0;
    case OP_SHUNT_LCP: /* Y = sC + 1/(sL) */
        nd[0] = 1; nd[1] = 0; nd[2] = p[0] * p[1] * wr2; nd[3] = 0; nd[4] = p[0] * wr; nd[5] = 0; return 0;
    default: return -1;
    }
}

/* Fused margin of one |S21| spec on a plain ladder (thread-per-sample kernel, qo_ts.cuh; its plan-time gate, qo_tf.cu):
 *     F(y) = N2(y) - t E(y)   (P.neg: fail where |den|^2 < t)      or      t E(y) - N2(y)   (fail where |den|^2 > t),
 * N2 = r0^2 - y r1^2 with r0 = sum_i cn[2i] y^i, r1 = sum_i cn[2i+1] y^i (kn pairs), E = sum_m ce[m] y^m (ke coefficients,
 * ke = 0: E = 1).  The sign of F is the verdict at a point, and F is one polynomial of max(2 kn, ke) coefficients.
 * Each coefficient is summed in double-double -- error-free products (fma(a, b, -a b)) and sums (two-sum), the low parts in
 * plain double -- and rounded once, so that it carries about one rounding whatever the cancellation between its terms.
 * Host and device run exactly this operation order (the products cannot be contracted: __dmul_rn on the device,
 * -ffp-contract=off on the host).  A zero F(0) coefficient is +0, so that F(y) is never -0 (an exact zero passes). */
QO_TF_HD double qo_tf_mul_rn(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
/* (s, c) += a b */
QO_TF_HD void qo_tf_dd_fma(double &s, double &c, double a, double b)
{
    const double p = qo_tf_mul_rn(a, b), pe = fma(a, b, -p);
    const double t = s + p, bp = t - s;
    c += ((s - (t - bp)) + (p - bp)) + pe;
    s = t;
}
/* coefficient k of F (the histogram screen of qo_ts.cuh forms them one at a time) */
QO_TF_HD double qo_tf_fuse_coef(int k, int kn, int ke, const double *cn, const double *ce, double t, bool neg)
{
    double s = 0.0, c = 0.0;
#pragma unroll
    for (int i = 0; i < kn; i++) {                        /* r0^2: a_i a_j (i + j = k), the off-diagonal pairs once, doubled */
        const int j = k - i;
        if (j >= i && j < kn) qo_tf_dd_fma(s, c, i == j ? cn[2 * i] : 2.0 * cn[2 * i], cn[2 * j]);
    }
#pragma unroll
    for (int i = 0; i < kn; i++) {                        /* - y r1^2: b_i b_j (i + j = k - 1) */
        const int j = k - 1 - i;
        if (j >= i && j < kn) qo_tf_dd_fma(s, c, i == j ? -cn[2 * i + 1] : -2.0 * cn[2 * i + 1], cn[2 * j + 1]);
    }
    if (k < (ke > 0 ? ke : 1)) qo_tf_dd_fma(s, c, -t, ke > 0 ? ce[k] : 1.0);
    const double v = s + c;
    return (neg ? v : -v) + 0.0;
}
QO_TF_HD void qo_tf_fuse(int kn, int ke, const double *cn, const double *ce, double t, bool neg, double *f)
{
    const int nf = 2 * kn > ke ? 2 * kn : ke;
#pragma unroll
    for (int k = 0; k < nf; k++) f[k] = qo_tf_fuse_coef(k, kn, ke, cn, ce, t, neg);
}

/* structural degree an element adds to the polynomials (max(deg N, deg D)); 0 = resistor, -1 = not lumped */
static inline int qo_tf_degree(int opcode)
{
    switch (opcode) {
    case OP_SER_R: case OP_SHUNT_G: return 0;
    case OP_SER_L: case OP_SHUNT_L: case OP_SER_C: case OP_SHUNT_C: return 1;
    case OP_SER_LOSSY_L: case OP_SHUNT_LOSSY_L: case OP_SER_LOSSY_C: case OP_SHUNT_LOSSY_C:
    case OP_SER_LCS: case OP_SER_LCP: case OP_SHUNT_LCS: case OP_SHUNT_LCP: return 2;
    default: return -1;
    }
}
