/* qo_ctx_internal.h -- device context shared by the CUDA translation units (qo_cuda.cu, qo_nodal.cu) */
#pragma once
#include <cuda_runtime.h>
#include "qo_internal.h"
#include "qo_tally.cuh"

/* a histogram request (cfg->hist_bins > 0) of a job with nspec specs: fits the counters, names one of the specs, has a window */
static inline bool qo_hist_cfg_ok(const qo_mc_cfg *cfg, int nspec)
{
    if (cfg->hist_bins <= QO_MAX_HIST && cfg->hist_spec >= 0 && cfg->hist_spec < nspec && cfg->hist_hi > cfg->hist_lo) return true;
    qo_set_error("bad histogram configuration");
    return false;
}

#define CU(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            qo_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));       \
            return (e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver) ? QO_ERR_NO_DEVICE : QO_ERR_CUDA; \
        }                                                                                             \
    } while (0)

/* ---- NCCL, loaded at run time (only the single-process multi-GPU ctx uses it) */
typedef struct ncclComm *ncclComm_t;
struct NcclApi {
    void *h;
    int (*CommInitAll)(ncclComm_t *, int, const int *);
    int (*CommDestroy)(ncclComm_t);
    int (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t);
    int (*GroupStart)(void);
    int (*GroupEnd)(void);
    const char *(*GetErrorString)(int);
};
struct DevCtx {
    int device;
    cudaStream_t stream;
    int own_stream;
    int sm_count;
    cudaEvent_t ev0, ev1;
};

struct qo_plan;
struct qo_ctx {
    int ndev;
    DevCtx d[8];
    NcclApi nccl;
    ncclComm_t comm[8];
    int have_nccl;
    /* the plan of the last qo_mc_run call, kept so that a caller who runs the same job again (a sweep over sample ranges, a
     * benchmark loop) does not rebuild the program, the polynomial analysis and the device allocation; its tables are still
     * copied host -> device on every call, one copy per device */
    struct qo_plan *mc_cache;
    unsigned long long mc_cache_key;
};

