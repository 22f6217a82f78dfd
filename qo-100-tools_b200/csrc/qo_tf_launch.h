/* qo_tf_launch.h -- host-visible entry points of the transfer-function kernel (qo_tf.cu) */
#pragma once
#include <cuda_runtime.h>
struct TfParams;
struct DevProg;
struct QoOverrides;
/* One run of the thread-per-sample kernel (qo_ts.cuh): consecutive groups of points that see the same spec bits, walked with
 * the polynomial lengths its own points need (never above the plan's kn / kd, the kernel's static capacities) */
#define QO_TS_MAXRUN 40          /* <= 4 band edges per spec, each at most one straddling group, plus the splits at length steps */
struct TsRun {
    int g0, ngroups;             /* first group, groups */
    unsigned int any, all;       /* spec bits seen by some / by every point of the run */
    int kn, ke;                  /* |numerator|^2 and E runs: numerator pairs and E coefficients walked (ke 0 without E) */
    int kf;                      /* runs of the fused spec: margin coefficients walked; runs of the histogram spec alone: coefficients
                                    of its screen walked (0: not screened); 0 on the other runs */
};
/* The histogram screen of the thread-per-sample kernel (qo_ts.cuh, plain ladders; its gate, qo_tf.cu::tf_hist_screen):
 * updates of the screen polynomial in place per sample, the plan's relative margin and its seed runs at most */
#define QO_TS_SCREEN_CAP 8
#define QO_TS_SCREEN_EPS 1e-6
#define QO_TS_NSEED 10
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
    /* the thread-per-sample kernel's run table (filled when qo_ts_eligible admits the job in some form): runs[0, ts_nplain) are
     * walked on |numerator|^2 and E, runs[ts_nplain, ts_nruns) are the fused spec's; ts_npt = the grid rounded up to whole
     * groups; ts_runs_ok = 0 when the band edges need more runs than the table holds */
    TsRun runs[QO_TS_MAXRUN];
    int ts_nruns, ts_nplain, ts_npt, ts_runs_ok;
    /* the histogram screen (runs with kf > 0 among the plain ones): its relative margin and the thresholds it covers, the seed runs
     * (the first ts_nseed runs: hist-band groups walked exactly before any screened one), the worst error bound the gate saw
     * relative to the margin, and "ok" or why the plan declined it */
    double ts_screen_eps, ts_screen_mlo, ts_screen_mhi, ts_screen_bound;
    int ts_nseed;
    const char *ts_screen_reason;
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
