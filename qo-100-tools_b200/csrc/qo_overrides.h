/*
 * qo_overrides.h -- the QO100NET_* environment overrides of the cascade (two-port) path and of the nodal (N-port) path, each
 * read in one place.
 *
 * qo_plan_create reads the cascade overrides once and keeps the record in the plan; everything that chooses a kernel reads the
 * record, never the environment.  qo_mc_run keys its plan cache, and qo_tf_plan_check its analysis cache, on the record's bytes,
 * so a new override changes both keys without a list of names to keep in step.  Every nodal entry point reads the nodal record
 * once per call.  Diagnostics and I/O switches (QO100NET_CHAIN_DEBUG, _CHAIN_JIT_DUMP, _NODAL_DEBUG, _NODAL_JIT_DUMP,
 * _CACHE_DIR, _NVRTC, _MC_TIMING, _NO_PLAN_CACHE) are read where they act.
 */
#pragma once
#include <stdlib.h>
#include <string.h>
#include "qo_internal.h"

struct QoOverrides {
    double tf_trunc;      /* QO100NET_TF_TRUNC: relative size of the polynomial terms the transfer-function analysis may drop */
    double tf_tol;        /* QO100NET_TF_TOL: tolerance of its self-check */
    enum Kernel { AUTO, TF, LADDER, INTERP } kernel;      /* QO100NET_KERNEL */
    int chain;            /* QO100NET_CHAIN: compiled chain kernel 1 always, -1 never, 0 by job size */
    int tf_no_front;      /* QO100NET_TF_NO_FRONT set: no line / measured two-port in front of the transfer-function kernel */
    int cpl_sincos;       /* QO100NET_CPL_SINCOS set: coupler angles by sincos per point, no table of nominal angles */
    int ustrip_item;      /* QO100NET_USTRIP=item: microstrip yield jobs on the item kernel, not thread-per-board */
    int ts_full_len;      /* QO100NET_TS_FULL_LENGTHS set: every run of the thread-per-sample kernel walks the plan's full polynomial lengths */
    int ts_no_screen;     /* QO100NET_TS_HIST_SCREEN=0: the thread-per-sample kernel walks the histogram band without its screen */
    int ts_low_seed;      /* QO100NET_TS_HIST_SEEDS=low: the band's lowest group is the screen's only seed (tests: the tracker then rises
                             after the seed, and the exact path moves the screen polynomial) */
};

/* QO_ERR_ARG (qo_last_error names the accepted values) when QO100NET_KERNEL holds anything but auto, spot, tf, ladder, interp */
static inline int qo_overrides_read(QoOverrides *ov)
{
    memset(ov, 0, sizeof *ov);            /* padding too: the caches hash the record's bytes */
    const char *k = getenv("QO100NET_KERNEL");
    if (!k || !*k || !strcmp(k, "auto") || !strcmp(k, "spot")) ov->kernel = QoOverrides::AUTO;
    else if (!strcmp(k, "tf")) ov->kernel = QoOverrides::TF;
    else if (!strcmp(k, "ladder")) ov->kernel = QoOverrides::LADDER;
    else if (!strcmp(k, "interp")) ov->kernel = QoOverrides::INTERP;
    else { qo_set_error("QO100NET_KERNEL=%s: expected auto, spot, tf, ladder or interp", k); return QO_ERR_ARG; }
    /* KERNEL=interp (A/B runs against the interpreter proper) also keeps the compiled chain kernel off unless CHAIN=jit says otherwise */
    const char *c = getenv("QO100NET_CHAIN");
    ov->chain = c && !strcmp(c, "jit") ? 1 : c && !strcmp(c, "interp") ? -1 : ov->kernel == QoOverrides::INTERP ? -1 : 0;
    const char *t = getenv("QO100NET_TF_TRUNC");
    ov->tf_trunc = t ? atof(t) : 5e-13;
    t = getenv("QO100NET_TF_TOL");
    ov->tf_tol = t ? atof(t) : 1e-10;
    ov->tf_no_front = getenv("QO100NET_TF_NO_FRONT") != NULL;
    ov->cpl_sincos = getenv("QO100NET_CPL_SINCOS") != NULL;
    const char *u = getenv("QO100NET_USTRIP");
    ov->ustrip_item = u && !strcmp(u, "item");
    ov->ts_full_len = getenv("QO100NET_TS_FULL_LENGTHS") != NULL;
    const char *hsc = getenv("QO100NET_TS_HIST_SCREEN");
    ov->ts_no_screen = hsc && !strcmp(hsc, "0");
    const char *hsd = getenv("QO100NET_TS_HIST_SEEDS");
    ov->ts_low_seed = hsd && !strcmp(hsd, "low");
    return QO_OK;
}

struct QoNodalOverrides {
    enum Kernel { AUTO, DENSE, STATIC, JIT } kernel;      /* QO100NET_NODAL */
    double growth2;       /* QO100NET_NODAL_GUARD2 above 0: the device's multiplier guard in place of QN_GROWTH2; else 0 */
};

/* QO_ERR_ARG (qo_last_error names the accepted values) when QO100NET_NODAL holds anything but auto, dense, static, jit */
static inline int qo_nodal_overrides_read(QoNodalOverrides *ov)
{
    memset(ov, 0, sizeof *ov);
    const char *k = getenv("QO100NET_NODAL");
    if (!k || !*k || !strcmp(k, "auto")) ov->kernel = QoNodalOverrides::AUTO;
    else if (!strcmp(k, "dense")) ov->kernel = QoNodalOverrides::DENSE;
    else if (!strcmp(k, "static")) ov->kernel = QoNodalOverrides::STATIC;
    else if (!strcmp(k, "jit")) ov->kernel = QoNodalOverrides::JIT;
    else { qo_set_error("QO100NET_NODAL=%s: expected auto, dense, static or jit", k); return QO_ERR_ARG; }
    const char *g = getenv("QO100NET_NODAL_GUARD2");      /* tests: trip the device guard on purpose */
    if (g && atof(g) > 0.0) ov->growth2 = atof(g);
    return QO_OK;
}
