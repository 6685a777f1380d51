// ihw.cu -- IHWcorrection(), "apply to test data" block (chicdiff.R:2038-2049), on the device.
//
// After R's ihw() has been trained on the control set and the distance lookup learned (:1994-2033), the test set gets, per
// region: group = cut(log|avDist|, breaks), weight = avWeights[group] / mean(avWeights over the rows),
// weighted_pvalue = pvalue / weight, weighted_padj = p.adjust(weighted_pvalue, "BH").  cd_ihw_apply (results.cpp) does
// that on the host (a stable sort of n p-values: ~0.3 s at 2 M regions); here the n-sized work runs on the GPU:
//   ihw_group_kernel    log|avDist|, binary search in the <= ngroups + 1 breaks, per-group counts (shared-memory histogram)
//   (host)              mean weight from the per-group counts, with R's long-double two-pass mean -- ngroups numbers, but
//                       n long-double additions, which the device has no type for (results_host.h: ihw_mean_weight)
//   ihw_weight_kernel   weight, weighted p-value, sort key
//   CUB radix sort      descending by weighted p-value, NA last
//   ihw_bh_value_kernel m / rank * p, then an inclusive minimum scan (CUB) = cummin from the largest p-value down
//   ihw_bh_write_kernel pmin(1, .) scattered back to input order
// Same arithmetic as the host routine operation by operation (m / rank * p, p / (w / mean)), so the two agree bit for
// bit wherever the device log and the host log put log|avDist| on the same side of a break.
#include "kernels.h"
#include "results_host.h"
#include <cub/cub.cuh>
#include <climits>
#include <vector>

namespace cd {

namespace {

constexpr int kIhwMaxSharedGroups = 1024;

__device__ __forceinline__ unsigned long long ihw_key(double x)           // order-preserving image; NaN -> 0 (sorts last descending)
{
    if (isnan(x)) return 0ull;
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double ihw_value(unsigned long long k)
{
    const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

__global__ void __launch_bounds__(256)
ihw_group_kernel(int64_t n, const double* __restrict__ avDist, const double* __restrict__ breaks, int ngroups,
                 int32_t* __restrict__ group, unsigned long long* __restrict__ counts /*ngroups + 1, [0] = NA*/)
{
    __shared__ unsigned int sh[kIhwMaxSharedGroups + 1];
    const bool use_sh = ngroups <= kIhwMaxSharedGroups;
    if (use_sh) {
        for (int k = threadIdx.x; k <= ngroups; k += blockDim.x) sh[k] = 0u;
        __syncthreads();
    }
    const double lo = breaks[0], hi = breaks[ngroups];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double x = log(fabs(avDist[i]));
        int32_t g = INT_MIN;                                              // NA_integer_
        if (!isnan(x) && x > lo && x <= hi) {
            // right-closed intervals (breaks[g-1], breaks[g]]: first break >= x
            int a = 0, b = ngroups;
            while (a < b) { const int m = (a + b) >> 1; if (breaks[m] < x) a = m + 1; else b = m; }
            g = a;
        }
        group[i] = g;
        const int slot = (g == INT_MIN) ? 0 : g;
        if (use_sh) atomicAdd(&sh[slot], 1u); else atomicAdd(counts + slot, 1ull);
    }
    if (use_sh) {
        __syncthreads();
        for (int k = threadIdx.x; k <= ngroups; k += blockDim.x)
            if (sh[k]) atomicAdd(counts + k, (unsigned long long)sh[k]);
    }
}

__global__ void __launch_bounds__(256)
ihw_weight_kernel(int64_t n, const int32_t* __restrict__ group, const double* __restrict__ pvalue,
                  const double* __restrict__ avWeights, double meanw, double* __restrict__ weight, double* __restrict__ wp,
                  unsigned long long* __restrict__ key, unsigned int* __restrict__ idx, unsigned long long* __restrict__ n_ok)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int ok = 0;
    if (i < n) {
        const int32_t g = group[i];
        const double w = (g == INT_MIN) ? NAN : avWeights[g - 1] / meanw;
        const double v = pvalue[i] / w;
        weight[i] = w;
        wp[i] = v;
        key[i] = ihw_key(v);
        idx[i] = (unsigned int)i;
        ok = isnan(v) ? 0u : 1u;
    }
    const unsigned int warp_ok = __popc(__ballot_sync(0xffffffffu, ok));
    if ((threadIdx.x & 31) == 0 && warp_ok) atomicAdd(n_ok, (unsigned long long)warp_ok);
}

// position t of the descending order holds rank m - t of the ascending one
__global__ void __launch_bounds__(256)
ihw_bh_value_kernel(int64_t n, const unsigned long long* __restrict__ key_sorted, const unsigned long long* __restrict__ n_ok,
                    double* __restrict__ v)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t m = (int64_t)*n_ok;
    v[t] = (t < m) ? (double)m / (double)(m - t) * ihw_value(key_sorted[t]) : INFINITY;
}

__global__ void __launch_bounds__(256)
ihw_bh_write_kernel(int64_t n, const unsigned int* __restrict__ idx_sorted, const unsigned long long* __restrict__ n_ok,
                    const double* __restrict__ cummin, double* __restrict__ padj)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int64_t m = (int64_t)*n_ok;
    // p.adjust returns a lone non-NA p-value unchanged, above 1 included
    padj[idx_sorted[t]] = (t < m) ? (m > 1 ? fmin(1.0, cummin[t]) : cummin[t]) : NAN;
}

struct Scratch {
    void* p = nullptr;
    ~Scratch() { if (p) cudaFree(p); }
    cudaError_t get(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
};

}  // namespace

// avDist_dev / pvalue_dev: n doubles in device memory.  Outputs: host arrays, any may be null.  Returns a CUDA error or,
// for the argument errors of the host routine, cudaErrorInvalidValue with *bad_breaks set.
cudaError_t ihw_apply_device(int64_t n, const double* avDist_dev, const double* pvalue_dev, int ngroups, const double* minLogDist,
                             const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                             double* weighted_pvalue_out, double* weighted_padj_out, bool* bad_breaks, cudaStream_t st)
{
    *bad_breaks = false;
    std::vector<double> breaks;
    if (!ihw_breaks(ngroups, minLogDist, maxLogDist, breaks)) { *bad_breaks = true; return cudaErrorInvalidValue; }
    if (n == 0) return cudaSuccess;
    if (n > (int64_t)INT_MAX) return cudaErrorInvalidValue;              // row indices are 32-bit; CUB counts in int
    const size_t nn = (size_t)n;
    Scratch s_breaks, s_w, s_counts, s_group, s_weight, s_wp, s_key, s_idx, s_v, s_tmp;
    cudaError_t e;
#define IHW_TRY(x) do { e = (x); if (e != cudaSuccess) return e; } while (0)
    IHW_TRY(s_breaks.get(sizeof(double) * ((size_t)ngroups + 1)));
    IHW_TRY(s_w.get(sizeof(double) * (size_t)ngroups));
    IHW_TRY(s_counts.get(sizeof(unsigned long long) * ((size_t)ngroups + 2)));
    IHW_TRY(s_group.get(sizeof(int32_t) * nn));
    IHW_TRY(s_weight.get(sizeof(double) * nn));
    IHW_TRY(s_wp.get(sizeof(double) * nn));
    IHW_TRY(s_key.get(sizeof(unsigned long long) * 2 * nn));
    IHW_TRY(s_idx.get(sizeof(unsigned int) * 2 * nn));
    IHW_TRY(s_v.get(sizeof(double) * 2 * nn));
    double* breaks_dev = (double*)s_breaks.p;
    double* w_dev = (double*)s_w.p;
    unsigned long long* counts = (unsigned long long*)s_counts.p;         // [0 .. ngroups]: per group; [ngroups + 1]: non-NA weighted p-values
    int32_t* group = (int32_t*)s_group.p;
    double *weight = (double*)s_weight.p, *wp = (double*)s_wp.p;
    unsigned long long *key0 = (unsigned long long*)s_key.p, *key1 = key0 + nn;
    unsigned int *idx0 = (unsigned int*)s_idx.p, *idx1 = idx0 + nn;
    double *v = (double*)s_v.p, *cummin = v + nn;
    IHW_TRY(cudaMemcpyAsync(breaks_dev, breaks.data(), sizeof(double) * ((size_t)ngroups + 1), cudaMemcpyHostToDevice, st));
    IHW_TRY(cudaMemcpyAsync(w_dev, avWeights, sizeof(double) * (size_t)ngroups, cudaMemcpyHostToDevice, st));
    IHW_TRY(cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * ((size_t)ngroups + 2), st));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned full = (unsigned)((n + 255) / 256);
    const unsigned capped = full < (unsigned)(sms * 8) ? full : (unsigned)(sms * 8);
    ihw_group_kernel<<<capped, 256, 0, st>>>(n, avDist_dev, breaks_dev, ngroups, group, counts);
    IHW_TRY(cudaGetLastError());
    std::vector<unsigned long long> per_group((size_t)ngroups + 1);
    IHW_TRY(cudaMemcpyAsync(per_group.data(), counts, sizeof(unsigned long long) * ((size_t)ngroups + 1), cudaMemcpyDeviceToHost, st));
    IHW_TRY(cudaStreamSynchronize(st));
    const double meanw = ihw_mean_weight(n, ngroups, per_group.data(), avWeights);
    ihw_weight_kernel<<<full, 256, 0, st>>>(n, group, pvalue_dev, w_dev, meanw, weight, wp, key0, idx0, counts + ngroups + 1);
    IHW_TRY(cudaGetLastError());
    if (group_out) IHW_TRY(cudaMemcpyAsync(group_out, group, sizeof(int32_t) * nn, cudaMemcpyDeviceToHost, st));
    if (weight_out) IHW_TRY(cudaMemcpyAsync(weight_out, weight, sizeof(double) * nn, cudaMemcpyDeviceToHost, st));
    if (weighted_pvalue_out) IHW_TRY(cudaMemcpyAsync(weighted_pvalue_out, wp, sizeof(double) * nn, cudaMemcpyDeviceToHost, st));
    if (weighted_padj_out) {
        size_t tmp_sort = 0, tmp_scan = 0;
        IHW_TRY(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_sort, key0, key1, idx0, idx1, (int)n, 0, 64, st));
        IHW_TRY(cub::DeviceScan::InclusiveScan(nullptr, tmp_scan, v, cummin, cub::Min(), (int)n, st));
        IHW_TRY(s_tmp.get(tmp_sort > tmp_scan ? tmp_sort : tmp_scan));
        IHW_TRY(cub::DeviceRadixSort::SortPairsDescending(s_tmp.p, tmp_sort, key0, key1, idx0, idx1, (int)n, 0, 64, st));
        ihw_bh_value_kernel<<<full, 256, 0, st>>>(n, key1, counts + ngroups + 1, v);
        IHW_TRY(cudaGetLastError());
        IHW_TRY(cub::DeviceScan::InclusiveScan(s_tmp.p, tmp_scan, v, cummin, cub::Min(), (int)n, st));
        ihw_bh_write_kernel<<<full, 256, 0, st>>>(n, idx1, counts + ngroups + 1, cummin, wp /* reused: padj in input order */);
        IHW_TRY(cudaGetLastError());
        IHW_TRY(cudaMemcpyAsync(weighted_padj_out, wp, sizeof(double) * nn, cudaMemcpyDeviceToHost, st));
    }
    IHW_TRY(cudaStreamSynchronize(st));
#undef IHW_TRY
    return cudaSuccess;
}

}  // namespace cd
