/*
 * qo_ustrip_board.cuh -- Qucs microstrip networks, one THREAD PER BOARD (sm_100a, FP64): reduce-only yield jobs at a handful
 * of frequencies (BASELINE config 3: util/pa-lpf-simulation/pa-lpf-simulation.sch:19-61 at the carrier and its harmonics,
 * pa-lpf-simulation.dpl:25-27; 1e7 boards x 3 points).
 *
 * qo_mc_generic_kernel (qo_ustrip.cuh) gives every (board, frequency) item its own thread, so with three frequencies per board
 *   - everything that does not depend on frequency -- the Hammerstad-Jensen quasi-static analysis of each strip width, about half
 *     of the Kirschning-Jansen dispersion terms, the loss and open-end constants: a third of the ~420 exp/log/atan/sincos calls of
 *     a point -- is computed three times, as are the board's variates and perturbed parameters;
 *   - each thread walks one long chain of dependent transcendental evaluations (ncu r02j: FP64 pipe 38.7 % busy, 39 % of the
 *     stall samples "wait", 16 warps per SM).
 * Here a thread owns a board and carries its NF frequencies through every model function side by side: the frequency-independent
 * part of a function runs once, the frequency-dependent part NF times in an unrolled loop of independent chains (ILP = NF), and
 * the ABCD chain is NF matrices wide.  The expressions are those of qo_ustrip.cuh term by term (same association, the hoisted
 * factors are exactly the sub-expressions the scalar code evaluates first), so a point's result differs from the scalar
 * kernel's by at most the compiler's FMA contraction choices; counters equal the oracle's (tests/test_gpu_parity.py).
 * Sweeps and FULL_S jobs (many frequencies per sample) stay on qo_mc_generic_kernel.
 */
#pragma once
#include "qo_ustrip.cuh"

#define QO_B_TPB 128
#ifndef QO_B_MINB
#define QO_B_MINB 3
#endif
#define QO_B_MAXNF 4
#define QO_BF _Pragma("unroll") for (int k = 0; k < NF; k++)

/* exp and log as CALLS: inlined, their ~190 expansions per frequency make this kernel 220 KB of code that every
 * warp streams through once per board (ncu r02k: 23 % of the stall samples "no instruction"); as small functions they stay in
 * the instruction cache (+15 % on config 3; sincos / cosh / sinh as calls, or the line section as a call, cost more than they
 * save).  The item-per-thread kernel keeps everything inline (calls cost it 10 %). */
__device__ __noinline__ double mb_exp(double x) { return exp(x); }
__device__ __noinline__ double mb_log(double x) { return ms_log(x); }
#define MB_POW(x, y) mb_exp((y) * mb_log(x))

/* Hammerstad-Jensen quasi-static line (ms_quasi with exp / log as calls) */
__device__ __noinline__ void ms_quasi_b(double W, const MsSub &s, double &Z, double &E, double &Weff)
{
    const double u = W / s.h;
    double du1 = 0.0, dur = 0.0;
    if (s.t > 0.0) {
        const double tau = s.t / s.h;
        const double th = tanh(sqrt(6.517 * u));
        du1 = (tau / QO_PI) * mb_log(1.0 + 4.0 * 2.7182818284590452354 * th * th / tau);
        dur = 0.5 * du1 * (1.0 + 1.0 / cosh(sqrt(s.er - 1.0)));
    }
    const double uu[2] = { u + dur, u + du1 };
    double zh[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const double x = uu[i];
        const double F = 6.0 + (2.0 * QO_PI - 6.0) * mb_exp(-MB_POW(30.666 / x, 0.7528));
        zh[i] = QO_ZF0 / (2.0 * QO_PI) * mb_log(F / x + sqrt(1.0 + 4.0 / (x * x)));
    }
    const double x = uu[0], x2 = x * x, x4 = x2 * x2;
    const double a = 1.0 + mb_log((x4 + x2 / 2704.0) / (x4 + 0.432)) / 49.0 + mb_log(1.0 + (x / 18.1) * (x / 18.1) * (x / 18.1)) / 18.7;
    const double b = 0.564 * MB_POW((s.er - 0.9) / (s.er + 3.0), 0.053);
    const double eps = 0.5 * (s.er + 1.0) + 0.5 * (s.er - 1.0) * MB_POW(1.0 + 10.0 / x, -a * b);
    const double ratio = zh[1] / zh[0];
    Z = zh[0] / sqrt(eps);
    E = eps * ratio * ratio;
    Weff = uu[0] * s.h;
}


/* MCORN(W): Kirschning-Jansen-Koster bend as a T network, SURVEY A.5 */
__device__ __noinline__ M2 ms_mcorn_b(double W, const MsSub &s, double f)
{
    const double wh = W / s.h;
    const double CpF = W * ((10.35 * s.er + 2.5) * wh + 2.6 * s.er + 5.64);
    const double LnH = 220.0 * s.h * (1.0 - 1.35 * mb_exp(-0.18 * MB_POW(wh, 1.39)));
    const double x21 = -0.5e12 / (QO_PI * f * CpF);          /* z21 = j x21 */
    const double x11 = 2e-9 * QO_PI * f * LnH + x21;          /* z11 = j x11 */
    M2 m;
    m.a = cmk(x11 / x21, 0.0);
    m.d = m.a;
    m.b = cmk(0.0, (x11 * x11 - x21 * x21) / x21);            /* (z11^2 - z21^2)/z21 = j (x11^2-x21^2)/x21 */
    m.c = cmk(0.0, -1.0 / x21);
    return m;
}



/* Kirschning-Jansen dispersion (ms_disp) for NF frequencies */
template <int NF>
__device__ __noinline__ void ms_disp_b(double W, const MsSub &s, double Z, double E, const double (&f)[NF], double (&Zf)[NF], double (&Ef)[NF])
{
    const double er = s.er, u = W / s.h;
    const double p1u = 0.065683 * mb_exp(-8.7513 * u);
    const double P2 = 0.33622 * (1.0 - mb_exp(-0.03442 * er));
    const double p3u = 0.0363 * mb_exp(-4.6 * u);
    const double P4 = 1.0 + 2.751 * (1.0 - mb_exp(-MB_POW(er / 15.916, 8.0)));
    const double R1 = 0.03891 * MB_POW(er, 1.4);
    const double R2 = 0.267 * MB_POW(u, 7.0);
    const double R3 = 4.766 * mb_exp(-3.228 * MB_POW(u, 0.641));
    const double R4 = 0.016 + MB_POW(0.0514 * er, 4.524);
    const double R6 = 22.20 * MB_POW(u, 1.92);
    const double R7 = 1.206 - 0.3144 * mb_exp(-R1) * (1.0 - mb_exp(-R2));
    const double c8 = -0.004625 * R3 * MB_POW(er, 1.674);
    const double e6 = MB_POW(er - 1.0, 6.0);
    const double a9 = 5.086 * R4, d4 = 0.3838 + 0.386 * R4, eR6 = mb_exp(-R6), d6 = 1.0 + 10.0 * e6;
    const double c15 = 0.707 * (0.00044 * MB_POW(er, 2.136) + 0.0184);
    const double c17 = 1.1241 * (1.0 / (1.0 + 0.00245 * u * u));
    const double c16 = 0.0503 * er * er, u15 = 1.0 - mb_exp(-MB_POW(u / 15.0, 6.0));
    QO_BF {
        const double fn = f[k] * s.h * 1e-6;
        const double P1 = 0.27488 + (0.6315 + 0.525 / MB_POW(1.0 + 0.0157 * fn, 20.0)) * u - p1u;
        const double P3 = p3u * (1.0 - mb_exp(-MB_POW(fn / 38.7, 4.97)));
        const double Pf = P1 * P2 * MB_POW((P3 * P4 + 0.1844) * fn, 1.5763);
        const double ef = er - (er - E) / (1.0 + Pf);
        Ef[k] = ef;
        const double R5 = MB_POW(fn / 28.843, 12.0);
        const double R8 = 1.0 + 1.275 * (1.0 - mb_exp(c8 * MB_POW(fn / 18.365, 2.745)));
        const double R9 = a9 * R5 / d4 * eR6 / (1.0 + 1.2992 * R5) * e6 / d6;
        const double t6 = MB_POW(fn / 19.47, 6.0);
        const double R11 = t6 / (1.0 + 0.0962 * t6);
        const double R13 = 0.9408 * MB_POW(ef, R8) - 0.9603;
        const double R14 = (0.9408 - R9) * MB_POW(E, R8) - 0.9603;
        const double R15 = c15 * MB_POW(fn / 12.3, 1.097);
        const double R16 = 1.0 + c16 * R11 * u15;
        const double R17 = R7 * (1.0 - c17 / R16 * mb_exp(-0.026 * MB_POW(fn, 1.15656) - R15));
        Zf[k] = Z * MB_POW(R13 / R14, R17);
    }
}

/* one strip width on this board: quasi-static values, and per frequency the dispersive Zf, Ef, sqrt(Ef) and the loss */
template <int NF> struct MsLineB { double W, Z, E, Weff, Zf[NF], Ef[NF], sq[NF], alpha[NF]; };
template <int NF> struct MsCacheB { MsLineB<NF> e[4]; int n, next; };

template <int NF>
__device__ __noinline__ void ms_line_fill_b(MsLineB<NF> &l, double W, const MsSub &s, const double (&f)[NF])
{
    l.W = W;
    ms_quasi_b(W, s, l.Z, l.E, l.Weff);
    ms_disp_b<NF>(W, s, l.Z, l.E, f, l.Zf, l.Ef);
    /* Hammerstad loss with the STATIC Z and E (SURVEY A.3) */
    const double Ki = mb_exp(-1.2 * MB_POW(l.Z / QO_ZF0, 0.7));
    const double zw = l.Z * W;
    const double cad = QO_PI * s.er / (s.er - 1.0) * (l.E - 1.0) / sqrt(l.E) * s.tand;
    QO_BF {
        const double Rs = sqrt(QO_PI * f[k] * QO_MU0 * s.rho);
        const double dd = s.D * Rs / s.rho;                 /* D / skin depth */
        const double Kr = 1.0 + (2.0 / QO_PI) * atan(1.4 * dd * dd);
        const double ac = Rs / zw * Ki * Kr;
        const double ad = cad * f[k] / QO_C0;
        l.alpha[k] = ac + ad;
        l.sq[k] = sqrt(l.Ef[k]);
    }
}

template <int NF>
__device__ __forceinline__ const MsLineB<NF> &ms_line_b(MsCacheB<NF> &c, double W, const MsSub &s, const double (&f)[NF])
{
    for (int i = 0; i < c.n; i++)
        if (c.e[i].W == W) return c.e[i];
    const int slot = c.n < 4 ? c.n++ : (c.next = (c.next + 1) & 3);
    ms_line_fill_b<NF>(c.e[slot], W, s, f);
    return c.e[slot];
}

/* MLIN(W, L) at the NF frequencies */
template <int NF>
__device__ __forceinline__ void ms_mlin_b(MsCacheB<NF> &c, double W, const double (&L)[NF], const MsSub &s, const double (&f)[NF], M2 (&m)[NF])
{
    const MsLineB<NF> &l = ms_line_b<NF>(c, W, s, f);
    double sb[NF], cb[NF], ch[NF], sh[NF];
    QO_BF {
        const double a = l.alpha[k] * L[k], b = 2.0 * QO_PI * f[k] * l.sq[k] / QO_C0 * L[k];
        sincos(b, &sb[k], &cb[k]);
        ch[k] = cosh(a); sh[k] = sinh(a);
    }
    QO_BF {
        m[k].a = cmk(ch[k] * cb[k], sh[k] * sb[k]);
        m[k].d = m[k].a;
        const cd shc = cmk(sh[k] * cb[k], ch[k] * sb[k]);
        m[k].b = cscale(shc, l.Zf[k]);
        m[k].c = cscale(shc, 1.0 / l.Zf[k]);
    }
}

/* MOPEN(W): B of Y = jB per frequency */
template <int NF>
__device__ __noinline__ void ms_mopen_b(MsCacheB<NF> &c, double W, const MsSub &s, const double (&f)[NF], double (&B)[NF])
{
    const MsLineB<NF> &l = ms_line_b<NF>(c, W, s, f);
    double Zf[NF], Ef[NF];
    ms_disp_b<NF>(l.Weff, s, l.Z, l.E, f, Zf, Ef);
    const double w = W / s.h, er = s.er;
    const double Q7 = MB_POW(w, 0.8544);
    const double Q2 = MB_POW(w, 0.371) / (2.358 * er + 1.0) + 1.0;
    const double q3 = atan(0.084 * MB_POW(w, 1.9413 / Q2)) * 0.5274;
    const double Q4 = 0.0377 * (6.0 - 5.0 * mb_exp(0.036 * (1.0 - er))) * atan(0.067 * MB_POW(w, 1.456)) + 1.0;
    const double Q5 = 1.0 - 0.218 * mb_exp(-7.5 * w);
    QO_BF {
        const double Q6 = MB_POW(Ef[k], 0.81);
        const double Q1 = 0.434907 * (Q6 + 0.26) / (Q6 - 0.189) * (Q7 + 0.236) / (Q7 + 0.87);
        const double Q3 = q3 / MB_POW(Ef[k], 0.9236) + 1.0;
        const double dl = Q1 * Q3 * Q5 / Q4 * s.h;
        B[k] = 2.0 * QO_PI * f[k] * dl * sqrt(Ef[k]) / (QO_C0 * Zf[k]);
    }
}

/* MTEE(Wa, Wb, W2) per frequency (ms_mtee) */
template <int NF>
__device__ __noinline__ void ms_mtee_b(MsCacheB<NF> &c, double Wa, double Wb, double W2, const MsSub &s, const double (&f)[NF], MsTee (&o)[NF])
{
    const MsLineB<NF> la = ms_line_b<NF>(c, Wa, s, f);
    const MsLineB<NF> lb = ms_line_b<NF>(c, Wb, s, f);
    const MsLineB<NF> l2 = ms_line_b<NF>(c, W2, s, f);
    const double h = s.h, er = s.er;
    QO_BF {
        const double fk = f[k];
        const double Da = QO_ZF0 / la.Zf[k] * h / la.sq[k], Db = QO_ZF0 / lb.Zf[k] * h / lb.sq[k], D2 = QO_ZF0 / l2.Zf[k] * h / l2.sq[k];
        const double fpa = 0.4e6 * la.Zf[k] / h, fpb = 0.4e6 * lb.Zf[k] / h;
        const double lda = QO_C0 / la.sq[k] / fk, ldb = QO_C0 / lb.sq[k] / fk;
        const double ra = la.Zf[k] / l2.Zf[k], rb = lb.Zf[k] / l2.Zf[k];
        const double fa2 = (fk / fpa) * (fk / fpa), fb2 = (fk / fpb) * (fk / fpb);
        const double da = 0.055 * D2 * ra * (1.0 - 2.0 * ra * fa2);
        const double db = 0.055 * D2 * rb * (1.0 - 2.0 * rb * fb2);
        o[k].La = 0.5 * W2 - da;
        o[k].Lb = 0.5 * W2 - db;
        const double r = sqrt(la.Zf[k] * lb.Zf[k]) / l2.Zf[k];
        const double q = fk * fk / (fpa * fpb);
        const double lr = mb_log(r);
        const double d2 = sqrt(Da * Db) * (0.5 - r * (0.05 + 0.7 * mb_exp(-1.6 * r) + 0.25 * r * q - 0.17 * lr));
        o[k].L2 = 0.5 * fmax(Wa, Wb) - d2;
        double ta = 1.0 - QO_PI * fa2 * (ra * ra / 12.0 + (0.5 - d2 / Da) * (0.5 - d2 / Da));
        double tb = 1.0 - QO_PI * fb2 * (rb * rb / 12.0 + (0.5 - d2 / Db) * (0.5 - d2 / Db));
        ta = fmax(ta, 1e-18);
        tb = fmax(tb, 1e-18);
        o[k].Ta2 = ta; o[k].Tb2 = tb;
        o[k].Bt = 5.5 * sqrt(Da * Db / (lda * ldb)) * (er + 2.0) / er / l2.Zf[k] / sqrt(ta * tb) * sqrt(da * db) / D2 *
                  (1.0 + 0.9 * lr + 4.5 * r * q - 4.4 * mb_exp(-1.3 * r) - 20.0 * (l2.Zf[k] / QO_ZF0) * (l2.Zf[k] / QO_ZF0));
    }
}

/* the full cascade of one board at its NF frequencies (qo_generic_abcd, NF matrices wide) */
template <int NF>
__device__ __forceinline__ void qo_board_abcd(const DevProg *__restrict__ prog, const double *x, const double (&f)[NF], M2 (&M)[NF])
{
    M2 Mmain[NF];
    QO_BF { M[k] = m2_ident(); Mmain[k] = m2_ident(); }
    MsSub sub = { 1.0, 1.0, 0.0, 0.0, 0.0, 0.0 };
    MsCacheB<NF> cache;
    cache.n = 0; cache.next = 3;
    MsTee tee[NF];
    QO_BF { tee[k].La = tee[k].Lb = tee[k].L2 = 0.0; tee[k].Ta2 = tee[k].Tb2 = 1.0; tee[k].Bt = 0.0; }
    double teeWa = 0.0, teeWb = 0.0;
    double cornW = -1.0, openW = -1.0, openB[NF], teeK[3] = { -1.0, -1.0, -1.0 };
    M2 cornM[NF];
    QO_BF { openB[k] = 0.0; cornM[k] = m2_ident(); }
    const int n_ops = prog->n_ops;
    for (int e = 0; e < n_ops; e++) {
        double p[6];
#pragma unroll
        for (int q = 0; q < 6; q++) {
            p[q] = prog->nom[e][q];
            const int tv = prog->tvar[e][q];
            if (tv >= 0) p[q] = qo_stream_apply(p[q], prog->ttol[e][q], x[tv], prog->tmode[e][q]);
        }
        const int kind = prog->kind[e];
        switch (kind) {
        case 1: QO_BF m2_series(M[k], cmk(p[0], 0.0)); break;
        case 2: QO_BF m2_shunt(M[k], cmk(1.0 / p[0], 0.0)); break;
        case 3: case 4:
            QO_BF {
                const double w = 2.0 * QO_PI * f[k];
                const cd z = cdiv(cmk(p[1], w * p[0]), cmk(1.0 - w * w * p[0] * p[2], w * p[1] * p[2]));
                if (kind == 3) m2_series(M[k], z); else m2_shunt(M[k], cinv(z));
            }
            break;
        case 5: case 6:
            QO_BF {
                const double w = 2.0 * QO_PI * f[k];
                const cd z = cmk(p[1], w * p[2] - 1.0 / (w * p[0]));
                if (kind == 5) m2_series(M[k], z); else m2_shunt(M[k], cinv(z));
            }
            break;
        case 7: QO_BF { const double w = 2.0 * QO_PI * f[k]; m2_series(M[k], cmk(0.0, w * p[0] - 1.0 / (w * p[1]))); } break;
        case 8: QO_BF { const double w = 2.0 * QO_PI * f[k]; m2_series(M[k], cmk(0.0, -1.0 / (w * p[1] - 1.0 / (w * p[0])))); } break;
        case 9: QO_BF { const double w = 2.0 * QO_PI * f[k]; m2_shunt(M[k], cmk(0.0, -1.0 / (w * p[0] - 1.0 / (w * p[1])))); } break;
        case 10: QO_BF { const double w = 2.0 * QO_PI * f[k]; m2_shunt(M[k], cmk(0.0, w * p[1] - 1.0 / (w * p[0]))); } break;
        case 11:
            QO_BF {
                const double w = 2.0 * QO_PI * f[k];
                double sn, cs;
                sincos(p[1] / 360.0 * w / p[2], &sn, &cs);
                M2 t;
                t.a = cmk(cs, 0.0); t.d = t.a; t.b = cmk(0.0, p[0] * sn); t.c = cmk(0.0, sn / p[0]);
                M[k] = m2_mul(M[k], t);
            }
            break;
        case 12: QO_BF M[k] = m2_mul(M[k], g_cpl(p, f[k])); break;
        case 13:
            sub.er = p[0]; sub.h = p[1]; sub.t = p[2]; sub.tand = p[3]; sub.rho = p[4]; sub.D = p[5];
            cache.n = 0;
            cornW = openW = teeK[0] = -1.0;
            break;
        case 14: {
            M2 t[NF];
            double L[NF];
            QO_BF L[k] = p[1];
            ms_mlin_b<NF>(cache, p[0], L, sub, f, t);
            QO_BF M[k] = m2_mul(M[k], t[k]);
            break;
        }
        case 15:
            if (p[0] != cornW) { QO_BF cornM[k] = ms_mcorn_b(p[0], sub, f[k]); cornW = p[0]; }
            QO_BF M[k] = m2_mul(M[k], cornM[k]);
            break;
        case 16: {
            if (p[0] != teeK[0] || p[1] != teeK[1] || p[2] != teeK[2]) {
                ms_mtee_b<NF>(cache, p[0], p[1], p[2], sub, f, tee);
                teeK[0] = p[0]; teeK[1] = p[1]; teeK[2] = p[2];
            }
            teeWa = p[0]; teeWb = p[1];
            double L[NF];
            QO_BF { Mmain[k] = M[k]; L[k] = tee[k].L2; }
            ms_mlin_b<NF>(cache, p[2], L, sub, f, M);        /* arm 2, junction outward */
            break;
        }
        case 17: {
            if (p[0] != openW) { ms_mopen_b<NF>(cache, p[0], sub, f, openB); openW = p[0]; }
            M2 ta[NF], tb[NF];
            double L[NF];
            QO_BF L[k] = tee[k].La;
            ms_mlin_b<NF>(cache, teeWa, L, sub, f, ta);
            QO_BF L[k] = tee[k].Lb;
            ms_mlin_b<NF>(cache, teeWb, L, sub, f, tb);
            QO_BF {
                const cd yo = cmk(0.0, openB[k]);
                const cd yin = cdiv(cadd(M[k].c, cmul(M[k].d, yo)), cadd(M[k].a, cmul(M[k].b, yo)));
                const double sa = sqrt(tee[k].Ta2), sb = sqrt(tee[k].Tb2);
                M2 m = m2_mul(Mmain[k], ta[k]);
                /* ideal transformers around the junction node and the shunt j Bt + Y_stub */
                m.a = cscale(m.a, 1.0 / sa); m.c = cscale(m.c, 1.0 / sa);
                m.b = cscale(m.b, sa); m.d = cscale(m.d, sa);
                m2_shunt(m, cmk(yin.re, yin.im + tee[k].Bt));
                m.a = cscale(m.a, sb); m.c = cscale(m.c, sb);
                m.b = cscale(m.b, 1.0 / sb); m.d = cscale(m.d, 1.0 / sb);
                M[k] = m2_mul(m, tb[k]);
            }
            break;
        }
        default: break;
        }
    }
}

/* one thread = one board; verdict and histogram per thread, counters through shared-memory atomics */
template <int NF>
__global__ void __launch_bounds__(QO_B_TPB, QO_B_MINB)
qo_mc_board_kernel(const DevProg *__restrict__ prog, const double *__restrict__ fgrid, const unsigned char *__restrict__ mask,
                   unsigned long long sample_offset, unsigned long long nsamples, unsigned long long *__restrict__ counters)
{
    __shared__ unsigned int s_cnt[QO_NCNT_MAX];
    const int nspec = prog->nspec, n_var = prog->n_var;
    const int hist_spec = prog->hist_bins > 0 ? prog->hist_spec : -1;
    const int hist_kind = hist_spec >= 0 ? prog->spec_user_kind[hist_spec] : 0;
    const bool hist_min = hist_kind == 1;     /* QO_SPEC_S21_MIN_DB: worst = smallest */
    const int ncnt = qo_ncnt(nspec, prog->hist_bins);
    qo_tally_zero<QO_B_TPB>(s_cnt, ncnt);
    __syncthreads();
    double f[NF];
    unsigned int mb[NF];
    QO_BF { f[k] = fgrid[k]; mb[k] = mask[k]; }
    for (unsigned long long s = (unsigned long long)blockIdx.x * QO_B_TPB + threadIdx.x; s < nsamples; s += (unsigned long long)gridDim.x * QO_B_TPB) {
        double x[QO_MAX_VAR];
        for (int v = 0; v < n_var; v++) x[v] = qo_stream_variate(prog->seed, sample_offset + s, (uint32_t)v, prog->dist);
        M2 M[NF];
        qo_board_abcd<NF>(prog, x, f, M);
        unsigned int fail = 0;
        unsigned long long worst = hist_min ? ~0ull : 0ull;
        QO_BF {
            cd s11, s21, s12, s22;
            qo_generic_s(prog, M[k], s11, s21, s12, s22);
            const double p21 = s21.re * s21.re + s21.im * s21.im, p11 = s11.re * s11.re + s11.im * s11.im;
            const double p22 = s22.re * s22.re + s22.im * s22.im;
            for (int sp = 0; sp < nspec; sp++) {
                if (!((mb[k] >> sp) & 1u)) continue;
                const int uk = prog->spec_user_kind[sp];
                const double lim = prog->spec_thr[sp];      /* linear power limit in this kernel */
                const double v = uk == 3 ? p11 : uk == 5 ? p22 : p21;      /* qo_spec_kind: |S11|, |S22|, else |S21| */
                const bool bad = uk == 1 ? (v < lim) : (v > lim);
                if (bad) fail |= 1u << sp;
                if (sp == hist_spec) {
                    const unsigned long long key = d2key(v);
                    worst = hist_min ? (key < worst ? key : worst) : (key > worst ? key : worst);
                }
            }
        }
        qo_tally_one(s_cnt, nspec, fail);
        if (hist_spec >= 0) {
            const double lin = __longlong_as_double((long long)worst);
            qo_tally_hist(s_cnt, nspec, qo_hist_bin(10.0 * log10(lin), prog->hist_lo, prog->hist_hi, prog->hist_bins));
        }
    }
    __syncthreads();
    qo_tally_flush<QO_B_TPB>(s_cnt, ncnt, counters);
}
