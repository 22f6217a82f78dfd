/*
 * qo_tally.cuh -- the counters every Monte-Carlo kernel returns, and the rule that bins a sample's histogram value.
 *
 * Layout, u32 per block in shared memory and u64 per job in global memory:
 *   [0] pass, [1] total, [2 + s] fails of spec s, [2 + nspec + b] samples in histogram bin b
 * A block zeroes its counters, tallies its samples into them with shared-memory atomics and adds them to the job's with one
 * global atomic per non-zero counter at the end; the barriers around that are the kernel's.
 *
 * Two habits keep the kernels' machine code what it was when each spelled this out itself (qo_mc_ts_kernel's SASS is the
 * profiled one): the thread index is read in the kernel, as a default argument -- read here it would carry no launch-bounds
 * range and, merged with the kernel's own read, take that range away -- and the job's scalars (nspec, the histogram window)
 * come by reference, so that a kernel's loads of P.nspec or prog->hist_bins stay where the kernel had them.
 *
 * Shared, as text, with the run-time compiled kernels (qo_chain_jit.h, qo_nodal_jit.h hand it to NVRTC), so it includes nothing.
 */
#ifndef QO_TALLY_CUH
#define QO_TALLY_CUH
#define QO_NSPEC_MAX 8
#define QO_MAX_HIST 1024
#define QO_NCNT_MAX (2 + QO_NSPEC_MAX + QO_MAX_HIST)

__host__ __device__ __forceinline__ int qo_ncnt(const int &nspec, const int &hist_bins) { return 2 + nspec + (hist_bins > 0 ? hist_bins : 0); }

/* bin = floor((v - lo) / (hi - lo) * bins); NaN and values below the window go to the first bin, values at or above it to the last */
__device__ __forceinline__ int qo_hist_bin(double v, const double &lo, const double &hi, const int &bins)
{
    const double xb = (v - lo) / (hi - lo) * (double)bins;
    long long b = (long long)floor(xb);
    if (!(xb >= 0.0)) b = 0;
    if (b >= bins) b = bins - 1;
    return (int)b;
}

template <int TPB> __device__ __forceinline__ void qo_tally_zero(unsigned int *cnt, int ncnt, int tid = threadIdx.x)
{
    for (int i = tid; i < ncnt; i += TPB) cnt[i] = 0;
}

/* one sample, recorded by one thread; fail: bit s set when the sample fails spec s */
__device__ __forceinline__ void qo_tally_one(unsigned int *cnt, const int &nspec, unsigned int fail)
{
    atomicAdd(&cnt[0], fail == 0 ? 1u : 0u);
    atomicAdd(&cnt[1], 1u);
    for (int sp = 0; sp < nspec; sp++)
        if ((fail >> sp) & 1u) atomicAdd(&cnt[2 + sp], 1u);
}

/* a warp's samples, one per lane, recorded by lane 0; vm: the lanes that hold a sample.  Called by all 32 lanes.  A constant
 * vm (0xffffffff: every lane holds one) costs no ballot for the total */
__device__ __forceinline__ void qo_tally_warp(unsigned int *cnt, const int &nspec, unsigned int fail, unsigned int vm, int lane = threadIdx.x & 31)
{
    const bool lane0 = lane == 0;
    const unsigned int pm = __ballot_sync(0xffffffffu, fail == 0u) & vm;
    if (lane0) { atomicAdd(&cnt[0], (unsigned int)__popc(pm)); atomicAdd(&cnt[1], (unsigned int)__popc(vm)); }
    for (int sp = 0; sp < nspec; sp++) {
        const unsigned int m = __ballot_sync(0xffffffffu, (fail >> sp) & 1u) & vm;
        if (lane0 && m) atomicAdd(&cnt[2 + sp], (unsigned int)__popc(m));
    }
}

/* one sample's histogram count, bin from qo_hist_bin */
__device__ __forceinline__ void qo_tally_hist(unsigned int *cnt, const int &nspec, int bin) { atomicAdd(&cnt[2 + nspec + bin], 1u); }

template <int TPB> __device__ __forceinline__ void qo_tally_flush(const unsigned int *cnt, int ncnt, unsigned long long *out, int tid = threadIdx.x)
{
    for (int i = tid; i < ncnt; i += TPB)
        if (cnt[i]) atomicAdd(&out[i], (unsigned long long)cnt[i]);
}
#endif
