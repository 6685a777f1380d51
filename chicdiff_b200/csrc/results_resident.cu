// results_resident.cu -- DESeq2 results() on the arrays the last cd_region_test left in device memory
// (chicdiff.R:1721,1730,1739; same rules as the host routine cd_results_adjust in results.cpp):
//   1. Cook's cutoff: p-value -> NA where maxCooks > qf(.99, p, m - p), unless the two-level heuristic kept the row
//   2. independent filtering: 50 baseMean quantile cut-offs (type 7), number of BH rejections at alpha for each
//   3. (host: lowess over the 50 counts and the threshold rule pick one cut-off)
//   4. BH adjusted p-values over the rows at or above that cut-off
// Everything global here is a sort: two radix sorts (baseMean keys; p-value keys carrying the row index), after
// which every cut-off is a prefix count over the p-sorted rows.  Chunks of 2048 sorted rows per CTA; the 50
// cut-offs share one load of the chunk.
#include "kernels.h"
#include "results_host.h"

namespace cd {

namespace {

constexpr int kResThreads = 256;
constexpr int kResItems = 8;
constexpr int kResChunk = kResThreads * kResItems;        // 2048 sorted rows per CTA
constexpr int kNT = 50;                                   // cut-offs tried by the independent filtering

__device__ __forceinline__ unsigned long long res_key(double x)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double res_value(unsigned long long k)
{
    const unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// Cook's filter + sort keys.  counts[0] = rows with a p-value, counts[1] = rows with baseMean == 0
__global__ void __launch_bounds__(256)
res_keys_kernel(int64_t n, int p, double cutoff, const double* __restrict__ baseMean, const double* __restrict__ maxCooks,
                const uint8_t* __restrict__ flags, const double* __restrict__ pvalue, double* __restrict__ pv_out,
                double* __restrict__ padj, unsigned long long* __restrict__ pkey, unsigned long long* __restrict__ bmkey,
                unsigned int* __restrict__ idx, unsigned long long* __restrict__ counts)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = false, zero = false;
    if (i < n) {
        double pv = pvalue[i];
        if (maxCooks[i] > cutoff) {                               // NaN compares false
            const bool keep = (flags[i] & CD_FLAG_COOKS_KEEP) && p == 2;
            if (!keep) pv = NAN;
        }
        const double bm = baseMean[i];
        valid = pv == pv;
        zero = bm == 0.0;
        pv_out[i] = pv;
        padj[i] = NAN;
        pkey[i] = valid ? res_key(pv) : ~0ull;
        bmkey[i] = res_key(bm);
        idx[i] = (unsigned int)i;
    }
    const unsigned bv = __ballot_sync(0xffffffffu, valid), bz = __ballot_sync(0xffffffffu, zero);
    if ((threadIdx.x & 31) == 0) {
        if (bv) atomicAdd(counts + 0, (unsigned long long)__popc(bv));
        if (bz) atomicAdd(counts + 1, (unsigned long long)__popc(bz));
    }
}

// quantile(baseMean, theta, type 7) for the 50 theta of genefilter's filtered_p call inside results(); lower and the
// index as R computes them (results_host.h)
__global__ void res_cutoffs_kernel(int64_t n, const unsigned long long* __restrict__ bm_sorted_keys,
                                   const unsigned long long* __restrict__ counts, double* __restrict__ cut /*50*/,
                                   double* __restrict__ theta_out /*50*/)
{
    const int k = threadIdx.x;
    if (k >= kNT) return;
    const double lower = n > 0 ? res_mean_of_count(counts[1], (uint64_t)n) : 0.0;
    const double upper = lower < .95 ? .95 : 1.0;
    const double step = __ddiv_rn(__dsub_rn(upper, lower), (double)(kNT - 1));
    const double theta = (k == kNT - 1) ? upper : __dadd_rn(lower, __dmul_rn((double)k, step));
    theta_out[k] = theta;
    if (n == 0) { cut[k] = NAN; return; }
    const ResQuantileIndex ix = res_quantile7_index(n, theta);
    double q = res_value(bm_sorted_keys[ix.lo]);
    const double qh = res_value(bm_sorted_keys[ix.hi]);
    if (ix.h > 0.0 && qh != q) q = __dadd_rn(__dmul_rn(__dsub_rn(1.0, ix.h), q), __dmul_rn(ix.h, qh));
    cut[k] = q;
}

// p-sorted order: baseMean and p-value of the row at each sorted position
__global__ void __launch_bounds__(256)
res_gather_kernel(int64_t n, const unsigned int* __restrict__ sorted_idx, const double* __restrict__ baseMean,
                  const double* __restrict__ pv, double* __restrict__ bm_s, double* __restrict__ p_s)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned int r = sorted_idx[i];
    bm_s[i] = baseMean[r];
    p_s[i] = pv[r];
}

// cnt[k * C + c] = rows of chunk c (sorted positions < nv) with baseMean >= cut[k]
__global__ void __launch_bounds__(kResThreads)
res_chunk_counts_kernel(const unsigned long long* __restrict__ counts, const double* __restrict__ bm_s,
                        const double* __restrict__ cut, int C, unsigned int* __restrict__ cnt)
{
    __shared__ double scut[kNT];
    __shared__ unsigned int tot[kNT];
    const int64_t nv = (int64_t)counts[0];
    const int c = blockIdx.x;
    if (threadIdx.x < kNT) { scut[threadIdx.x] = cut[threadIdx.x]; tot[threadIdx.x] = 0u; }
    __syncthreads();
    double bm[kResItems];
    const int64_t base = (int64_t)c * kResChunk + (int64_t)threadIdx.x * kResItems;
#pragma unroll
    for (int j = 0; j < kResItems; j++) bm[j] = (base + j < nv) ? bm_s[base + j] : NAN;       // NaN >= x is false
    for (int k = 0; k < kNT; k++) {
        unsigned int m = 0;
#pragma unroll
        for (int j = 0; j < kResItems; j++) m += (bm[j] >= scut[k]) ? 1u : 0u;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m += __shfl_down_sync(0xffffffffu, m, off);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&tot[k], m);
    }
    __syncthreads();
    if (threadIdx.x < kNT) cnt[(size_t)threadIdx.x * C + c] = tot[threadIdx.x];
}

// per cut-off: exclusive prefix over the chunks (in place) and the total m[k]
__global__ void __launch_bounds__(256)
res_chunk_scan_kernel(int C, unsigned int* __restrict__ cnt, unsigned long long* __restrict__ m_out /*50*/)
{
    __shared__ unsigned long long part[256];
    const int k = blockIdx.x;
    unsigned int* a = cnt + (size_t)k * C;
    const int per = (C + 255) / 256;
    const int lo = threadIdx.x * per, hi = min(C, lo + per);
    unsigned long long s = 0;
    for (int c = lo; c < hi; c++) s += a[c];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int t = 0; t < 256; t++) { const unsigned long long v = part[t]; part[t] = run; run += v; }
        m_out[k] = run;
    }
    __syncthreads();
    unsigned long long run = part[threadIdx.x];
    for (int c = lo; c < hi; c++) { const unsigned int v = a[c]; a[c] = (unsigned int)run; run += v; }
}

// block-wide exclusive prefix sum of one unsigned per thread (kResThreads threads); every thread gets its offset
__device__ __forceinline__ unsigned int block_excl_sum(unsigned int v, unsigned int* warp_tot /*shared, 8*/)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned int o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    __syncthreads();                                  // warp_tot may still be read from the previous call
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    unsigned int before = 0;
    for (int w = 0; w < wid; w++) before += warp_tot[w];
    return before + inc - v;
}

// best[k] = largest rank r (among the rows with baseMean >= cut[k], in ascending p order) with m/r * p < alpha
__global__ void __launch_bounds__(kResThreads)
res_num_rej_kernel(const unsigned long long* __restrict__ counts, const double* __restrict__ bm_s, const double* __restrict__ p_s,
                   const double* __restrict__ cut, int C, const unsigned int* __restrict__ off /*50 x C*/,
                   const unsigned long long* __restrict__ m_tot /*50*/, double alpha, unsigned long long* __restrict__ best /*50*/)
{
    __shared__ double scut[kNT];
    __shared__ unsigned int warp_tot[kResThreads / 32];
    const int64_t nv = (int64_t)counts[0];
    const int c = blockIdx.x;
    if (threadIdx.x < kNT) scut[threadIdx.x] = cut[threadIdx.x];
    __syncthreads();
    double bm[kResItems], pv[kResItems];
    const int64_t base = (int64_t)c * kResChunk + (int64_t)threadIdx.x * kResItems;
#pragma unroll
    for (int j = 0; j < kResItems; j++) {
        const bool in = base + j < nv;
        bm[j] = in ? bm_s[base + j] : NAN;
        pv[j] = in ? p_s[base + j] : NAN;
    }
    for (int k = 0; k < kNT; k++) {
        unsigned int mine = 0;
#pragma unroll
        for (int j = 0; j < kResItems; j++) mine += (bm[j] >= scut[k]) ? 1u : 0u;
        const unsigned int before = block_excl_sum(mine, warp_tot);
        const double m = (double)m_tot[k];
        unsigned long long rank = (unsigned long long)off[(size_t)k * C + c] + before, local = 0;
#pragma unroll
        for (int j = 0; j < kResItems; j++) {
            if (!(bm[j] >= scut[k])) continue;
            rank++;
            if (m / (double)rank * pv[j] < alpha) local = rank;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long x = __shfl_down_sync(0xffffffffu, local, o);
            local = x > local ? x : local;
        }
        if ((threadIdx.x & 31) == 0 && local) atomicMax(best + k, local);
    }
}

// BH at cut-off j, step 1: v = m / rank * p per kept row; minimum of every chunk
__global__ void __launch_bounds__(kResThreads)
res_bh_chunk_min_kernel(const unsigned long long* __restrict__ counts, const double* __restrict__ bm_s,
                        const double* __restrict__ p_s, const double* __restrict__ cut, int j, int C,
                        const unsigned int* __restrict__ off, const unsigned long long* __restrict__ m_tot,
                        double* __restrict__ cmin /*C*/)
{
    __shared__ unsigned int warp_tot[kResThreads / 32];
    __shared__ double wmin[kResThreads / 32];
    const int64_t nv = (int64_t)counts[0];
    const int c = blockIdx.x;
    const double cj = cut[j], m = (double)m_tot[j];
    double bm[kResItems], pv[kResItems];
    const int64_t base = (int64_t)c * kResChunk + (int64_t)threadIdx.x * kResItems;
    unsigned int mine = 0;
#pragma unroll
    for (int q = 0; q < kResItems; q++) {
        const bool in = base + q < nv;
        bm[q] = in ? bm_s[base + q] : NAN;
        pv[q] = in ? p_s[base + q] : NAN;
        mine += (bm[q] >= cj) ? 1u : 0u;
    }
    const unsigned int before = block_excl_sum(mine, warp_tot);
    unsigned long long rank = (unsigned long long)off[(size_t)j * C + c] + before;
    double lo = INFINITY;
#pragma unroll
    for (int q = 0; q < kResItems; q++) {
        if (!(bm[q] >= cj)) continue;
        rank++;
        lo = fmin(lo, m / (double)rank * pv[q]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lo = fmin(lo, __shfl_down_sync(0xffffffffu, lo, o));
    if ((threadIdx.x & 31) == 0) wmin[threadIdx.x >> 5] = lo;
    __syncthreads();
    if (threadIdx.x == 0) {
        double x = wmin[0];
        for (int w = 1; w < kResThreads / 32; w++) x = fmin(x, wmin[w]);
        cmin[c] = x;
    }
}

// step 2: smin[c] = min over the chunks after c (exclusive suffix minimum); one CTA
__global__ void __launch_bounds__(256)
res_bh_suffix_kernel(int C, const double* __restrict__ cmin, double* __restrict__ smin)
{
    __shared__ double part[256];
    const int per = (C + 255) / 256;
    const int lo = threadIdx.x * per, hi = min(C, lo + per);
    double x = INFINITY;
    for (int c = lo; c < hi; c++) x = fmin(x, cmin[c]);
    part[threadIdx.x] = x;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = INFINITY;
        for (int t = 255; t >= 0; t--) { const double v = part[t]; part[t] = run; run = fmin(run, v); }
    }
    __syncthreads();
    double run = part[threadIdx.x];
    for (int c = hi - 1; c >= lo; c--) { smin[c] = run; run = fmin(run, cmin[c]); }
}

// step 3: running minimum from the largest p-value down, capped at 1, scattered to the rows
__global__ void __launch_bounds__(kResThreads)
res_bh_write_kernel(const unsigned long long* __restrict__ counts, const double* __restrict__ bm_s, const double* __restrict__ p_s,
                    const unsigned int* __restrict__ sorted_idx, const double* __restrict__ cut, int j, int C,
                    const unsigned int* __restrict__ off, const unsigned long long* __restrict__ m_tot,
                    const double* __restrict__ smin, double* __restrict__ padj)
{
    __shared__ unsigned int warp_tot[kResThreads / 32];
    __shared__ double tmin[kResThreads];
    const int64_t nv = (int64_t)counts[0];
    const int c = blockIdx.x;
    const double cj = cut[j], m = (double)m_tot[j];
    double bm[kResItems], v[kResItems];
    const int64_t base = (int64_t)c * kResChunk + (int64_t)threadIdx.x * kResItems;
    unsigned int mine = 0;
#pragma unroll
    for (int q = 0; q < kResItems; q++) {
        const bool in = base + q < nv;
        bm[q] = in ? bm_s[base + q] : NAN;
        v[q] = in ? p_s[base + q] : NAN;
        mine += (bm[q] >= cj) ? 1u : 0u;
    }
    const unsigned int before = block_excl_sum(mine, warp_tot);
    unsigned long long rank = (unsigned long long)off[(size_t)j * C + c] + before;
    double lo = INFINITY;
#pragma unroll
    for (int q = 0; q < kResItems; q++) {
        if (!(bm[q] >= cj)) { v[q] = INFINITY; continue; }
        rank++;
        v[q] = m / (double)rank * v[q];
        lo = fmin(lo, v[q]);
    }
    // exclusive suffix minimum over the threads after this one (Hillis-Steele on shared memory), then the later chunks
    tmin[threadIdx.x] = lo;
    __syncthreads();
    for (int o = 1; o < kResThreads; o <<= 1) {
        const double other = (threadIdx.x + o < kResThreads) ? tmin[threadIdx.x + o] : INFINITY;
        __syncthreads();
        tmin[threadIdx.x] = fmin(tmin[threadIdx.x], other);
        __syncthreads();
    }
    double run = (threadIdx.x + 1 < kResThreads) ? tmin[threadIdx.x + 1] : INFINITY;
    run = fmin(run, smin[c]);
#pragma unroll
    for (int q = kResItems - 1; q >= 0; q--) {
        if (!(bm[q] >= cj)) continue;
        run = fmin(run, v[q]);
        padj[sorted_idx[base + q]] = fmin(1.0, run);
    }
}

inline unsigned nblk(int64_t n) { return (unsigned)((n + 255) / 256); }

}  // namespace

cudaError_t res_launch_keys(int64_t n, int p, double cutoff, const double* baseMean, const double* maxCooks, const uint8_t* flags,
                            const double* pvalue, double* pv_out, double* padj, unsigned long long* pkey,
                            unsigned long long* bmkey, unsigned int* idx, unsigned long long* counts, cudaStream_t st)
{
    cudaError_t e = cudaMemsetAsync(counts, 0, 2 * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    if (n > 0)
        res_keys_kernel<<<nblk(n), 256, 0, st>>>(n, p, cutoff, baseMean, maxCooks, flags, pvalue, pv_out, padj, pkey, bmkey, idx, counts);
    return cudaGetLastError();
}

cudaError_t res_launch_cutoffs(int64_t n, const unsigned long long* bm_sorted_keys, const unsigned long long* counts, double* cut,
                               double* theta, cudaStream_t st)
{
    res_cutoffs_kernel<<<1, 64, 0, st>>>(n, bm_sorted_keys, counts, cut, theta);
    return cudaGetLastError();
}

cudaError_t res_launch_gather(int64_t n, const unsigned int* sorted_idx, const double* baseMean, const double* pv, double* bm_s,
                              double* p_s, cudaStream_t st)
{
    if (n > 0) res_gather_kernel<<<nblk(n), 256, 0, st>>>(n, sorted_idx, baseMean, pv, bm_s, p_s);
    return cudaGetLastError();
}

int res_chunks(int64_t n) { return (int)((n + kResChunk - 1) / kResChunk); }

cudaError_t res_launch_num_rej(int64_t n, const unsigned long long* counts, const double* bm_s, const double* p_s,
                               const double* cut, unsigned int* cnt, unsigned long long* m_tot, double alpha,
                               unsigned long long* best, cudaStream_t st)
{
    const int C = res_chunks(n);
    cudaError_t e = cudaMemsetAsync(best, 0, kNT * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    if (C == 0) return cudaMemsetAsync(m_tot, 0, kNT * sizeof(unsigned long long), st);
    res_chunk_counts_kernel<<<C, kResThreads, 0, st>>>(counts, bm_s, cut, C, cnt);
    res_chunk_scan_kernel<<<kNT, 256, 0, st>>>(C, cnt, m_tot);
    res_num_rej_kernel<<<C, kResThreads, 0, st>>>(counts, bm_s, p_s, cut, C, cnt, m_tot, alpha, best);
    return cudaGetLastError();
}

cudaError_t res_launch_bh(int64_t n, const unsigned long long* counts, const double* bm_s, const double* p_s,
                          const unsigned int* sorted_idx, const double* cut, int j, const unsigned int* off,
                          const unsigned long long* m_tot, double* cmin, double* smin, double* padj, cudaStream_t st)
{
    const int C = res_chunks(n);
    if (C == 0) return cudaSuccess;
    res_bh_chunk_min_kernel<<<C, kResThreads, 0, st>>>(counts, bm_s, p_s, cut, j, C, off, m_tot, cmin);
    res_bh_suffix_kernel<<<1, 256, 0, st>>>(C, cmin, smin);
    res_bh_write_kernel<<<C, kResThreads, 0, st>>>(counts, bm_s, p_s, sorted_idx, cut, j, C, off, m_tot, smin, padj);
    return cudaGetLastError();
}

}  // namespace cd
