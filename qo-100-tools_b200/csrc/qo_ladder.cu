/*
 * qo_ladder.cu -- instantiations and launcher of the straight-line ladder kernel
 * (qo_ladder.cuh).  Its own translation unit so that the 44 instantiations
 * (N = 1..11, series/shunt first, with/without the coupled-line block) compile
 * in parallel with qo_cuda.cu.
 */
#include <cuda_runtime.h>
#include "qo_ladder.cuh"
#include "qo_ladder_launch.h"

/* launch shape chosen from the r01 ncu sweeps (DESIGN.md "ladder kernel"): */
#ifndef QO_LAD_PP
#define QO_LAD_PP 2
#define QO_LAD_TPB 256
#define QO_LAD_MINB 2
#endif

typedef void (*lad_fn)(const LadParams);

template <typename T, int N, int FIRST, bool CPL, int NROWS, int PP, int TPB, int MINB> static lad_fn lad_get()
{
    return qo_mc_ladder_kernel<T, N, FIRST, CPL, NROWS, PP, TPB, MINB>;
}

template <typename T, int NROWS, int PP, int TPB, int MINB> static lad_fn lad_pick(int n, int first, int cpl)
{
#define QO_LAD_ROW(NN)                                                                       \
    case NN:                                                                                 \
        return cpl ? (first ? lad_get<T, NN, 1, true, NROWS, PP, TPB, MINB>() : lad_get<T, NN, 0, true, NROWS, PP, TPB, MINB>())   \
                   : (first ? lad_get<T, NN, 1, false, NROWS, PP, TPB, MINB>() : lad_get<T, NN, 0, false, NROWS, PP, TPB, MINB>());
    switch (n) {
        QO_LAD_ROW(1) QO_LAD_ROW(2) QO_LAD_ROW(3) QO_LAD_ROW(4) QO_LAD_ROW(5) QO_LAD_ROW(6)
        QO_LAD_ROW(7) QO_LAD_ROW(8) QO_LAD_ROW(9) QO_LAD_ROW(10) QO_LAD_ROW(11)
    default: return nullptr;
    }
#undef QO_LAD_ROW
}

/* kernels with the |S11| row: two points per thread (the second row vector doubles the chain state) */
#define QO_LAD2_PP 1
#define QO_LAD2_TPB 256
#define QO_LAD2_MINB 2

typedef void (*lad_fn_t)(const LadParams);
extern "C" lad_fn_t qo_ladder_pick32(int n, int first, int cpl, int *tpb, int *minb);

extern "C" int qo_ladder_launch(int n, int first, int cpl, int nrows, int precision, int sm_count, const LadParams *P, cudaStream_t st)
{
    lad_fn fn;
    int tpb, minb;
    if (precision == 32) {
        if (nrows != 1) return -1;
        fn = qo_ladder_pick32(n, first, cpl, &tpb, &minb);      /* qo_ladder32.cu */
    } else if (nrows == 2) {
        fn = lad_pick<double, 2, QO_LAD2_PP, QO_LAD2_TPB, QO_LAD2_MINB>(n, first, cpl);
        tpb = QO_LAD2_TPB; minb = QO_LAD2_MINB;
    } else {
        fn = lad_pick<double, 1, QO_LAD_PP, QO_LAD_TPB, QO_LAD_MINB>(n, first, cpl);
        tpb = QO_LAD_TPB; minb = QO_LAD_MINB;
    }
    if (!fn) return -1;
    const unsigned long long warps = (unsigned long long)(tpb / 32);
    unsigned long long blocks = (P->nsamples + warps - 1) / warps;
    const unsigned long long resident = (unsigned long long)sm_count * (unsigned long long)minb;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    fn<<<(unsigned)blocks, tpb, 0, st>>>(*P);
    return (int)cudaGetLastError();
}
