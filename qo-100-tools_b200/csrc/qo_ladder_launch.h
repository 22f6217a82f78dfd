/* qo_ladder_launch.h -- host-visible launcher of the straight-line ladder kernel (qo_ladder.cu) */
#pragma once
#include <cuda_runtime.h>
struct LadParams;
/* returns 0, -1 when no instantiation covers (n, first, cpl), else the cudaError_t of the launch */
extern "C" int qo_ladder_launch(int n, int first, int cpl, int nrows, int precision, int sm_count, const LadParams *P, cudaStream_t st);
