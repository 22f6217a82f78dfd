/* qo_tf_launch.h -- host-visible entry points of the transfer-function kernel (qo_tf.cu) */
#pragma once
#include <cuda_runtime.h>
struct TfParams;
struct DevProg;
struct QoOverrides;
/* what the plan decided for a job that runs on the transfer-function kernel */
struct TfPlan {
    int nn;              /* numerator chains: 2 (Num = P + Rs Q) or 4 (P and Q apart: behind a coupled-line block, or with |S11| specs) */
    int s11;             /* the job has |S11| specs */
    int gd;              /* the job has group-delay specs (derivative polynomials ride along) */
    int den;             /* QO_TF_DEN_* */
    int kn, kd;          /* coefficient pairs kept per numerator polynomial; E coefficients (even count) or D pairs kept */
    int deg;             /* structural degree of the numerator polynomials */
    int el0, n_el;       /* the lumped ops */
    int cpl_op;          /* the block in front of the lumped ops (its row vector is contracted with [P; Q] per point), -1 = none */
    int front;           /* what that block is: 0 coupled-line section, 1 transmission line (OP_TLINE), 2 measured two-port (OP_SBLOCK) */
    double wref;         /* normalising angular frequency (geometric centre of the grid) */
    double err;          /* worst relative disagreement on |den|^2 seen by the self-check */
    unsigned int fused;  /* specs whose single-spec runs the thread-per-sample kernel walks on the fused margin (qo_tf_fuse) */
    double fused_err;    /* worst disagreement of the fused margin with the unfused one, relative to |den|^2 (over every spec tried) */
    const char *reason;  /* "ok", or why the job stays on the chain kernels */
};
/* Can this job run on the transfer-function kernel?  Structural test, choice of the polynomial lengths the grid needs,
 * and a numerical self-check of exactly what the device will evaluate against the per-element evaluation, at the
 * nominal network and at both ends of its tolerance box, on every grid point.  Returns 1 (plan filled) or 0. */
extern "C" int qo_tf_plan_check(const DevProg *hp, int mode_reduce_only, int precision, int generic, const double *f, int nf,
                                const unsigned char *mask, const QoOverrides *ov, TfPlan *out);
/* pp = frequency pairs per thread per iteration the plan padded its tables for; returns 0, -1 when no
 * instantiation covers (nn, den, pp), else the cudaError_t of the launch */
extern "C" int qo_tf_launch(const TfPlan *tp, int pp, int sm_count, const TfParams *P, cudaStream_t st);
extern "C" int qo_tf_default_pp(const TfPlan *tp, int npairs);

/* thread-per-sample flavour (qo_ts.cuh): eligibility, threads per wave, launch (0 or the cudaError_t) */
struct TsParams;
extern "C" int qo_ts_eligible(const TfPlan *tp, int nspec, int cpl_rot_same);
extern "C" int qo_ts_wave_threads(const TfPlan *tp, int sm_count);
extern "C" int qo_ts_group_points(const TfPlan *tp);
extern "C" int qo_ts_launch(const TfPlan *tp, int sm_count, const TsParams *Q, cudaStream_t st);

/* spot-frequency kernel (qo_spot.cuh): one thread per sample, <= 8 frequencies; returns 0 or the cudaError_t of the launch */
struct SpotParams;
extern "C" int qo_spot_launch(int need_s11, int sm_count, const SpotParams *P, cudaStream_t st);

/* FULL_S flavour of the transfer-function kernel (qo_tf_fs.cuh) */
struct TfFsParams;
extern "C" int qo_tf_fs_plan_check(const DevProg *hp, int mode_full_s, int precision, int generic, const double *f, int nf, const QoOverrides *ov,
                                   TfPlan *out);
extern "C" int qo_tf_fs_launch(int dmode, int sm_count, const TfFsParams *P, cudaStream_t st);   /* dmode: 0 D == 1, 1 polynomial D, 2 factored D */
