/*
 * qo_device.cuh -- device-side program layout shared by the kernels and the host
 * plan builder.
 *
 * A network is compiled on the host into a flat "program": one opcode per
 * element plus, per (element, parameter), the random variable that perturbs it.
 * Per Monte-Carlo sample the kernels derive a table of *hoisted coefficients*
 * (1/C, L*Cp, R*Cp, ...) once, stage it in shared memory, and every thread then
 * evaluates its own (sample, frequency) points against that table.
 */
#pragma once
#include <stdint.h>
#include "qo_tally.cuh"      /* QO_NSPEC_MAX, QO_MAX_HIST */

#define QO_MAX_OPS 96
#define QO_MAX_VAR 64
#define QO_MAX_COEF 256      /* doubles per per-sample coefficient table */

enum {
    OP_NOP = 0,
    OP_SER_R, OP_SHUNT_G,
    OP_SER_L, OP_SER_C, OP_SER_LCS,          /* series, purely imaginary: X = w*c0 - winv*c1 */
    OP_SHUNT_C, OP_SHUNT_L, OP_SHUNT_LCP,    /* shunt,  purely imaginary: B = w*c0 - winv*c1 */
    OP_SER_LCP,                              /* series parallel-LC tank:  X = -1/(w*C - winv/L) */
    OP_SHUNT_LCS,                            /* shunt series-LC trap:     B = -1/(w*L - winv/C) */
    OP_SER_LOSSY_L, OP_SHUNT_LOSSY_L,        /* (L, L*Cp, R, R*Cp) */
    OP_SER_LOSSY_C, OP_SHUNT_LOSSY_C,        /* (1/C, Ls, R, R*R)  */
    OP_TLINE,                                /* (Z0, 1/Z0, theta/w) */
    OP_CPL,                                  /* (z0e/zt, zt/z0e, z0o/zt, zt/z0o, te/w, to/w, zt, 1/zt) */
    OP_SBLOCK,                               /* (block index): per-frequency ABCD table of a measured two-port */
    /* distributed microstrip opcodes: generic kernel only */
    OP_SUBST, OP_MLIN, OP_MCORN, OP_MTEE, OP_MOPEN
};

/* canonical spec forms: a point FAILS when q > thr */
enum { SK_DEN2_MAX = 1 /* S21_MIN_DB: |den|^2 <= thr */, SK_DEN2_MIN = 2 /* S21_MAX_DB: |den|^2 >= thr */,
       SK_S11_MAX = 3 /* |n11|^2 <= thr*|den|^2 */, SK_GD_MAX = 4, SK_S22_MAX = 5 /* |n22|^2 <= thr*|den|^2 */ };
//@mu{ lines between these markers reach the run-time compiled chain kernel's source only for jobs with a stability spec
enum { SK_MU_MIN = 6 /* Edwards-Sinsky mu = num / den with den >= 0: a point fails when !(num >= thr*den) */ };
//@mu}

struct DevProg {
    int32_t n_ops, n_var, n_coef, dist;
    int32_t nspec, hist_spec, hist_bins, need_s11;
    int32_t has_trig, has_ustrip, need_gd, op0;     /* op0: first op that is not an OP_NOP (a SUBST that only serves a QO_CPL_MS) */
    int32_t cplms_elem, cplms_sub;                  /* physical coupled-line element and its substrate element, -1 = none */
    int32_t need_s22, pad2;                         /* need_s22 sits where a pad was: every other field keeps its offset */
    double cplms_nom[4];                            /* its nominal Z0e, Z0o, theta_e, theta_o [deg] */
    uint64_t seed;
    double rs, rl, rsrl, k21;                /* k21 = 2*sqrt(rs*rl) */
    double hist_lo, hist_hi;                 /* bin = floor((v - lo) / (hi - lo) * bins) */
    int32_t spec_kind[QO_NSPEC_MAX];         /* SK_* */
    int32_t spec_user_kind[QO_NSPEC_MAX];    /* qo_spec_kind */
    double spec_thr[QO_NSPEC_MAX];           /* canonical (linear) threshold */
    double spec_limit[QO_NSPEC_MAX];         /* user limit (dB / s) */
    int32_t opcode[QO_MAX_OPS];
    int32_t coff[QO_MAX_OPS];                /* offset of the op's coefficients */
    int32_t kind[QO_MAX_OPS];                /* qo_kind of the source element */
    double nom[QO_MAX_OPS][6];
    double ttol[QO_MAX_OPS][6];
    int16_t tvar[QO_MAX_OPS][6];             /* -1 = not perturbed */
    uint8_t tmode[QO_MAX_OPS][6];            /* 0 REL, 1 ABS */
};
