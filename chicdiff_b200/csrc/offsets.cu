// offsets.cu -- size factors, the parametric dispersion trend of a batch of fits, and the deterministic
// reductions the global steps need.
//
//   chicdiff.R:1561-1562  estimateSizeFactors: log-ratio matrix (medians by radix selection, select.cu)
//   DESeq2 momentsDispEstimate: mean over samples of 1 / colMeans(normalisation factors of the non-zero rows)
//   DESeq2 parametricDispersionFit / dispersionFunction<-: Gamma(identity) IRLS sums, fitted
//                         trend and log residuals
//   chicdiff.R:1647       sum of deviances per theta-grid fit
//
// (the per-region normalisation offsets of stage 2, chicdiff.R:1583-1589 / 1614-1615 / 1635-1638, are in
// dispersion.cu: norm_factors_kernel writes them for every fit of a batch.)
//
// All reductions are two-stage with a fixed block count and fixed summation order, so results
// are bit-reproducible from run to run (no floating-point atomics).
#include "kernels.h"

namespace cd {

static inline int blocks_for(int64_t n, int threads) { return (int)((n + threads - 1) / threads); }

constexpr long long kSpinLimit = 20000000000LL;      // ~10 s of SM clocks: a peer died; give up

template <int NV>
__device__ __forceinline__ void block_reduce_store(double (&v)[NV], double* dst)
{
    __shared__ double sh[NV][8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; k++) {
        double x = v[k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
        if (lane == 0) sh[k][wid] = x;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double x = 0.0;
        const int nw = blockDim.x >> 5;
        for (int w = 0; w < nw; w++) x += sh[threadIdx.x][w];
        dst[threadIdx.x] = x;
    }
    __syncthreads();
}

// final stage: out[k] = sum_b partial[b*nv + k]; one warp per value, lanes stride over the blocks
// and a fixed shuffle tree joins them, so the summation order never changes
__global__ void __launch_bounds__(32) final_reduce_kernel(int nblocks, int nv, const double* __restrict__ partial,
                                                          double* __restrict__ out)
{
    const int k = blockIdx.x;
    double x = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += 32) x += partial[(size_t)b * nv + k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x += __shfl_down_sync(0xffffffffu, x, off);
    if (threadIdx.x == 0) out[k] = x;
}

// ---------------------------------------------------------------------------------------
// masked column sums per fit of a batch: M is sample-major over the G * n virtual regions;
// out[g * (S + 1) + s] = sum over the rows of fit g with mask == 0 of M[s][.] ; out[g * (S + 1) + S] = #rows
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
masked_colsums_kernel(int64_t n, int G, int S, const double* __restrict__ M, const uint8_t* __restrict__ mask,
                      double* __restrict__ partial)
{
    const int64_t nv = (int64_t)G * n;
    const int64_t chunk = (n + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * chunk;
    const int64_t hi = (lo + chunk < n) ? lo + chunk : n;
    for (int g = 0; g < G; g++)
        for (int s = 0; s <= S; s++) {
            double v[1] = {0.0};
            for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
                const int64_t r = (int64_t)g * n + i;
                const bool use = (mask == nullptr) || ((mask[r] & CD_FLAG_ALLZERO) == 0);
                if (use) v[0] += (s < S) ? M[(int64_t)s * nv + r] : 1.0;
            }
            block_reduce_store<1>(v, partial + ((size_t)blockIdx.x * G + g) * (S + 1) + s);
        }
}

cudaError_t launch_masked_colsums(int64_t n, int G, int S, const double* M, const uint8_t* mask, double* partial,
                                  double* out, cudaStream_t st)
{
    masked_colsums_kernel<<<kReduceBlocks, 256, 0, st>>>(n, G, S, M, mask, partial);
    final_reduce_kernel<<<G * (S + 1), 32, 0, st>>>(kReduceBlocks, G * (S + 1), partial, out);
    return cudaGetLastError();
}

// out[g] = sum of v over the rows of fit g (NaN propagates: chicdiff.R:1647 sums without na.rm)
__global__ void __launch_bounds__(256)
segment_sums_kernel(int64_t n, int G, const double* __restrict__ v_in, double* __restrict__ partial)
{
    const int64_t chunk = (n + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * chunk;
    const int64_t hi = (lo + chunk < n) ? lo + chunk : n;
    for (int g = 0; g < G; g++) {
        double v[1] = {0.0};
        for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) v[0] += v_in[(int64_t)g * n + i];
        block_reduce_store<1>(v, partial + (size_t)blockIdx.x * G + g);
    }
}

cudaError_t launch_segment_sums(int64_t n, int G, const double* v, double* partial, double* out, cudaStream_t st)
{
    segment_sums_kernel<<<kReduceBlocks, 256, 0, st>>>(n, G, v, partial);
    final_reduce_kernel<<<G, 32, 0, st>>>(kReduceBlocks, G, partial, out);
    return cudaGetLastError();
}

// xim[g] = mean_s 1 / (colsum_s / count)   (momentsDispEstimate), sums laid out as masked_colsums writes them
__global__ void xim_kernel(int G, int S, const double* __restrict__ sums, double* __restrict__ xim)
{
    const int g = threadIdx.x;
    if (g >= G) return;
    const double* sg = sums + (size_t)g * (S + 1);
    const double cnt = sg[S];
    double acc = 0.0;
    for (int s = 0; s < S; s++) acc += 1.0 / (sg[s] / cnt);
    xim[g] = acc / S;
}

cudaError_t launch_xim(int G, int S, const double* sums, double* xim, cudaStream_t st)
{
    xim_kernel<<<1, 32, 0, st>>>(G, S, sums, xim);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// size factors: LR[s][i] = log K[s][i] - mean_s' log K[s'][i] for rows with every K > 0,
// +inf otherwise (excluded from the medians).  This is the one pass of a region test that reads every count, so it
// also checks them: DESeqDataSetFromMatrix (chicdiff.R:1556-1559) refuses NA (NA_integer_ = INT32_MIN, what the
// aggregation writes for a sum beyond the int32 range) and negative counts; *bad = 1.0 tells the host to do the same.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
log_ratios_kernel(int64_t n, int S, const int32_t* __restrict__ K, double* __restrict__ LR, double* __restrict__ bad)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc = 0.0;
    bool ok = true, neg = false;
    for (int s = 0; s < S; s++) {
        const int32_t k = K[(int64_t)s * n + i];
        ok = ok && (k > 0);
        neg = neg || (k < 0);
        acc += log((double)k);
    }
    if (neg) *bad = 1.0;                       // every writer stores the same value: no atomic needed
    const double lgm = acc / S;
    for (int s = 0; s < S; s++)
        LR[(int64_t)s * n + i] = ok ? log((double)K[(int64_t)s * n + i]) - lgm : INFINITY;
}

cudaError_t launch_log_ratios(int64_t n, int S, const int32_t* K, double* LR, double* bad, cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    log_ratios_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, S, K, LR, bad);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// The whole parametricDispersionFit of a batch of G fits on the device: one cooperative kernel, one CTA per SM.
// Every pass (sums + deviance at coefficients b over the rows kept by the outer coefficients c, for every fit that
// is still running) is a chunked block reduction, a grid barrier, and a fixed-order sum of the per-CTA partials
// that every CTA repeats for itself, so all CTAs take the same branch of glm.fit's control flow (start validity,
// IRLS <= 25, step halving, outer loop <= 11) without a host round trip.  Thread g of every CTA runs fit g's control
// flow; the G fits advance in lock step, so a batch costs max_g(passes) barriers, not their sum.
// out[g * 8 + 0..1] = coefficients, [2] = status (0 ok; 1..5 = reason the reference would fall back to a local fit;
// 6 = the exchange with another rank failed), [3] = outer iterations, [4] = passes.
// ---------------------------------------------------------------------------------------
constexpr int kTrendThreads = 512;
constexpr int kTrendSlot = 8 * kMaxBatch + 8;      // doubles per mailbox slot: 8 sums per fit, then the sequence word

__device__ __forceinline__ bool trend_grid_barrier(unsigned int* bar, unsigned int nblocks, unsigned int& phase,
                                                   unsigned long long* err)
{
    __shared__ int ok_sh;
    __syncthreads();
    phase++;                                   // every thread keeps the same phase count
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
        int ok = 1;
        const long long t0 = clock64();
        while (atomicAdd(bar, 0u) < phase * nblocks) {
            if (*reinterpret_cast<volatile unsigned long long*>(err) != 0ull) { ok = 0; break; }
            if (clock64() - t0 > kSpinLimit) { ok = 0; atomicExch(err, 1ull); break; }
        }
        __threadfence();
        ok_sh = ok;
    }
    __syncthreads();
    return ok_sh != 0;
}

// Cross-GPU part of a pass (sharded runs): CTA 0 stores this rank's sums straight into every peer's mailbox over
// NVLink, then a sequence word.  EVERY CTA then waits until all ranks' slots of the local mailbox carry this pass's
// sequence and adds them in rank order, so all CTAs of all ranks obtain bit-identical totals and follow the same
// control flow, without a second grid barrier.  Slots are double-buffered by pass parity: a peer can only be one pass
// ahead, because finishing a pass needs everybody's contribution to it, and CTA 0 contributes to pass k+1 only after
// the grid barrier of pass k+1, i.e. after all local CTAs have read pass k.  A CTA that gives up raises the error
// word, which ends every other spin loop (here and in the grid barrier) of this and of the following kernels.
constexpr int kTrendMaxRanks = 16;                   // peer-memory mailboxes exist for up to 16 ranks (cd_comm_init)
__device__ __forceinline__ bool p2p_allreduce(const TrendP2P& pp, unsigned long long seq, unsigned int parity, int nvals,
                                              double* sh_tot)
{
    __shared__ int timed_out;
    if (threadIdx.x == 0) timed_out = 0;
    __syncthreads();
    if (blockIdx.x == 0) {
        for (int r = 0; r < pp.nranks; r++) {
            double* dst = pp.peers[r] + ((size_t)parity * pp.nranks + pp.rank) * kTrendSlot;
            for (int k = threadIdx.x; k < nvals; k += blockDim.x) dst[k] = sh_tot[k];
        }
        __threadfence_system();
        __syncthreads();
        if ((int)threadIdx.x < pp.nranks) {
            double* dst = pp.peers[threadIdx.x] + ((size_t)parity * pp.nranks + pp.rank) * kTrendSlot;
            *reinterpret_cast<volatile unsigned long long*>(dst + 8 * kMaxBatch) = seq;
        }
    }
    if ((int)threadIdx.x < pp.nranks) {
        volatile unsigned long long* f = reinterpret_cast<volatile unsigned long long*>(
            pp.mymail + ((size_t)parity * pp.nranks + threadIdx.x) * kTrendSlot + 8 * kMaxBatch);
        const long long t0 = clock64();
        while (*f != seq) {
            if (*reinterpret_cast<volatile unsigned long long*>(pp.err) != 0ull) { timed_out = 1; break; }
            if (clock64() - t0 > kSpinLimit) { timed_out = 1; atomicExch(pp.err, 1ull); break; }
        }
        __threadfence_system();
        // how long this rank waited for the slowest peer's sums (CTA 0, per peer): the rendezvous cost the bench reports
        // ([2]: the part of [0] spent in the first pass of a launch, which absorbs the ranks' different arrival times)
        if (blockIdx.x == 0 && pp.wait_cycles) {
            const unsigned long long w = (unsigned long long)(clock64() - t0);
            atomicAdd(pp.wait_cycles + ((int)threadIdx.x == pp.rank ? 1 : 0), w);
            if ((int)threadIdx.x != pp.rank && (seq & 0xffffffffull) == 1ull) atomicAdd(pp.wait_cycles + 2, w);
        }
    }
    __syncthreads();
    if ((int)threadIdx.x < nvals) {
        // the slots are final once the sequence words are seen: L2 loads, all in flight, summed in rank order
        double v[kTrendMaxRanks];
#pragma unroll
        for (int r = 0; r < kTrendMaxRanks; r++)
            v[r] = (r < pp.nranks) ? __ldcg(pp.mymail + ((size_t)parity * pp.nranks + r) * kTrendSlot + threadIdx.x) : 0.0;
        double x = 0.0;
#pragma unroll
        for (int r = 0; r < kTrendMaxRanks; r++)
            if (r < pp.nranks) x += v[r];
        sh_tot[threadIdx.x] = x;
    }
    __syncthreads();
    return timed_out == 0;
}

// what one pass evaluates for one fit
struct TrendPass { double c0, c1, b0, b1; int refresh, active; };

// glm.fit's control flow for one fit, advanced by one pass at a time (thread g of every CTA holds fit g's copy)
struct TrendFit {
    double c0, c1, b0, b1, ob0, ob1, nb0, nb1, devold;
    double v[8];
    int iter, it, halv, passes, status, stage;       // stage 0: first pass of an outer iteration, 1: IRLS proposal, 2: done
    bool conv;

    __device__ void init()
    {
        c0 = 0.1; c1 = 1.0; b0 = c0; b1 = c1; ob0 = c0; ob1 = c1; nb0 = c0; nb1 = c1; devold = 0.0;
        iter = 0; it = 0; halv = 0; passes = 0; status = 0; stage = 0; conv = false;
    }
    __device__ void next_pass(TrendPass& p) const
    {
        p.c0 = c0; p.c1 = c1;
        p.active = (stage != 2);
        if (stage == 0) { p.b0 = c0; p.b1 = c1; p.refresh = (passes == 0) ? 2 : 1; }
        else { p.b0 = nb0; p.b1 = nb1; p.refresh = 0; }
    }
    __device__ void propose()
    {
        const double det = v[0] * v[2] - v[1] * v[1];
        nb0 = (v[2] * v[3] - v[1] * v[4]) / det;
        nb1 = (v[0] * v[4] - v[1] * v[3]) / det;
        halv = 0;
    }
    __device__ void outer_end()
    {
        const double oc0 = c0, oc1 = c1;
        c0 = b0; c1 = b1;
        if (!(c0 > 0.0 && c1 > 0.0)) { status = 4; stage = 2; return; }
        const double l0 = log(c0 / oc0), l1 = log(c1 / oc1);
        if ((l0 * l0 + l1 * l1 < 1e-6) && conv) { stage = 2; return; }
        iter++;
        if (iter > 10) { status = 5; stage = 2; return; }
        stage = 0;
    }
    // w: the 8 totals of the pass that next_pass() described
    __device__ void advance(const double* w)
    {
        passes++;
        if (stage == 0) {
            b0 = c0; b1 = c1; ob0 = c0; ob1 = c1;
#pragma unroll
            for (int k = 0; k < 8; k++) v[k] = w[k];
            if (v[7] < 2.0) { status = 1; stage = 2; return; }
            if (v[6] > 0.0) { status = 2; stage = 2; return; }
            devold = v[5]; conv = false; it = 0;
            propose();
            stage = 1;
            return;
        }
        if (!(w[6] == 0.0 && isfinite(w[5]))) {
            if (++halv > 25) { status = 3; stage = 2; return; }
            nb0 = 0.5 * (nb0 + ob0); nb1 = 0.5 * (nb1 + ob1);
            return;
        }
        b0 = nb0; b1 = nb1;
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = w[k];
        const double dev = w[5];
        if (fabs(dev - devold) / (fabs(dev) + 0.1) < 1e-8) { conv = true; outer_end(); return; }
        devold = dev; ob0 = b0; ob1 = b1;
        if (++it < 25) { propose(); return; }
        outer_end();
    }
};

// One pass for one fit: the sums glm.fit needs at coefficients b over the rows kept by the outer coefficients c.
// xs is scratch (one double per virtual region) that carries 1/baseMean between passes: NaN = row never used (all-zero
// region or dispersion at the floor), negative = excluded by the current outer coefficients.  refresh = 2 on the first
// pass of the launch (fill xs), 1 on the first pass of an outer iteration (re-decide the sign), 0 otherwise.
// Every row is always handled by the same thread, so xs needs no synchronisation.
__device__ __forceinline__ void trend_row(int64_t i, double d, double xv, int refresh, double c0, double c1, double b0, double b1,
                                          double* __restrict__ xs, double (&v)[8])
{
    if (refresh) {
        if (xv != xv) { if (refresh == 2) xs[i] = xv; return; }
        const double x = fabs(xv);
        const double r = d / (c0 + c1 * x);
        xv = ((r > 1e-4) && (r < 15.0)) ? x : -x;
        xs[i] = xv;
    }
    if (!(xv > 0.0)) return;
    const double x = xv;
    const double mu = b0 + b1 * x;
    v[7] += 1.0;
    if (!(mu > 0.0) || !isfinite(mu)) { v[6] += 1.0; return; }
    double w, t;
    if (mu > 1e-100 && mu < 1e100) { const double inv = rcp_pos(mu); w = inv * inv; t = d * inv; }
    else { w = 1.0 / (mu * mu); t = d / mu; }
    const double wx = w * x;
    v[0] += w; v[1] += wx; v[2] += wx * x;
    v[3] += w * d; v[4] += wx * d;
    // unit deviance of the Gamma family: -2 (log(d/mu) - (d - mu)/mu)
    const double lt = (t > 1e-300 && t < 1e300) ? log_pos(t) : log(t);
    v[5] += -2.0 * (lt - (t - 1.0));
}

// The pass streams 16 bytes per row; four rows per thread are loaded before any of them is processed so that enough
// loads are in flight to cover the HBM latency (a thread handles the same rows, in the same order, in every pass, so
// the sums stay bit-reproducible).
__device__ __forceinline__ void trend_pass_rows(int64_t lo, int64_t hi, const double* __restrict__ baseMean,
                                                const double* __restrict__ dispGeneEst, const uint8_t* __restrict__ flags,
                                                double* __restrict__ xs, const TrendPass& p, double (&v)[8])
{
    const int refresh = p.refresh;
    const double c0 = p.c0, c1 = p.c1, b0 = p.b0, b1 = p.b1;
    const int64_t bd = blockDim.x;
    int64_t i = lo + threadIdx.x;
    for (; i + 3 * bd < hi; i += 4 * bd) {
        double d[4], xv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) d[u] = dispGeneEst[i + u * bd];
        if (refresh == 2) {
            double bm[4];
            uint8_t f[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { bm[u] = baseMean[i + u * bd]; f[u] = flags[i + u * bd]; }
#pragma unroll
            for (int u = 0; u < 4; u++) xv[u] = (!(f[u] & CD_FLAG_ALLZERO) && (d[u] > 100.0 * kMinDisp)) ? 1.0 / bm[u] : NAN;
        } else {
#pragma unroll
            for (int u = 0; u < 4; u++) xv[u] = xs[i + u * bd];
        }
#pragma unroll
        for (int u = 0; u < 4; u++) trend_row(i + u * bd, d[u], xv[u], refresh, c0, c1, b0, b1, xs, v);
    }
    for (; i < hi; i += bd) {
        const double d = dispGeneEst[i];
        double xv;
        if (refresh == 2) xv = (!(flags[i] & CD_FLAG_ALLZERO) && (d > 100.0 * kMinDisp)) ? 1.0 / baseMean[i] : NAN;
        else xv = xs[i];
        trend_row(i, d, xv, refresh, c0, c1, b0, b1, xs, v);
    }
}

__global__ void __launch_bounds__(kTrendThreads)
trend_fit_kernel(int64_t n, int G, const double* __restrict__ baseMean, const double* __restrict__ dispGeneEst,
                 const uint8_t* __restrict__ flags, double* __restrict__ xs, double* partial, unsigned int* bar, double* out,
                 TrendP2P pp)
{
    __shared__ double tot[8 * kMaxBatch];
    __shared__ double shw[8 * kMaxBatch][kTrendThreads / 32];
    __shared__ TrendPass sp[kMaxBatch];
    __shared__ int any_active, failed;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nvals = 8 * G;
    unsigned int phase = 0;
    unsigned long long pass_no = 0;
    TrendFit fit;
    fit.init();
    if (threadIdx.x == 0) failed = 0;
    const int64_t chunk = (n + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * chunk;
    const int64_t hi = (lo + chunk < n) ? lo + chunk : n;
    while (true) {
        if ((int)threadIdx.x < G) fit.next_pass(sp[threadIdx.x]);
        if (threadIdx.x == 0) any_active = 0;
        __syncthreads();
        if ((int)threadIdx.x < G && sp[threadIdx.x].active) any_active = 1;
        __syncthreads();
        if (!any_active) break;
        // partials are double-buffered by pass parity: a CTA can be at most one pass ahead of the slowest
        // one (there is a barrier in every pass), so one barrier per pass is enough
        double* part = partial + (size_t)(phase & 1u) * nvals * gridDim.x;
        for (int g = 0; g < G; g++) {
            double v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (sp[g].active) {
                const int64_t off = (int64_t)g * n;
                trend_pass_rows(off + lo, off + hi, baseMean, dispGeneEst, flags, xs, sp[g], v);
            }
#pragma unroll
            for (int k = 0; k < 8; k++) {
                double x = v[k];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
                if (lane == 0) shw[g * 8 + k][wid] = x;
            }
        }
        __syncthreads();
        if ((int)threadIdx.x < nvals) {
            double x = 0.0;
            for (int w = 0; w < kTrendThreads / 32; w++) x += shw[threadIdx.x][w];
            __stcg(part + (size_t)blockIdx.x * nvals + threadIdx.x, x);
        }
        bool ok = trend_grid_barrier(bar, gridDim.x, phase, pp.err);
        if (ok) {
            // fixed-order sum of the per-CTA partials, one warp per value; every CTA repeats it for itself
            for (int k = wid; k < nvals; k += kTrendThreads / 32) {
                double x = 0.0;
                for (unsigned b = lane; b < gridDim.x; b += 32) x += __ldcg(part + (size_t)b * nvals + k);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
                if (lane == 0) tot[k] = x;
            }
            __syncthreads();
            if (pp.nranks > 1) {
                pass_no++;
                ok = p2p_allreduce(pp, (pp.epoch << 32) | pass_no, (unsigned int)(pass_no & 1ull), nvals, tot);
            }
        }
        if (!ok) {
            if (threadIdx.x == 0) failed = 1;
            __syncthreads();
            break;
        }
        if ((int)threadIdx.x < G && sp[threadIdx.x].active) fit.advance(tot + 8 * threadIdx.x);
        __syncthreads();
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < G) {
        double* o = out + 8 * threadIdx.x;
        o[0] = fit.c0; o[1] = fit.c1; o[2] = failed ? 6.0 : (double)fit.status; o[3] = (double)(fit.iter + 1);
        o[4] = (double)fit.passes;
    }
}

cudaError_t launch_trend_fit(int64_t n, int G, const double* baseMean, const double* dispGeneEst, const uint8_t* flags,
                             double* xs, double* partial, unsigned int* bar, double* out, const TrendP2P& pp_in, cudaStream_t st)
{
    if (G < 1 || G > kMaxBatch) return cudaErrorInvalidValue;
    TrendP2P pp = pp_in;
    int dev = 0, sms = 148, coop = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    if (!coop) return cudaErrorNotSupported;
    cudaError_t e = cudaMemsetAsync(bar, 0, sizeof(unsigned int), st);
    if (e != cudaSuccess) return e;
    void* args[] = {(void*)&n, (void*)&G, (void*)&baseMean, (void*)&dispGeneEst, (void*)&flags, (void*)&xs, (void*)&partial, (void*)&bar,
                    (void*)&out, (void*)&pp};
    return cudaLaunchCooperativeKernel((const void*)trend_fit_kernel, dim3((unsigned)sms), dim3(kTrendThreads), args, 0, st);
}

// dispFit = a0 + a1/baseMean ; resid = log(dispGeneEst) - log(dispFit) or +inf when excluded ; coefs[g * 8 + 0..1] on device
__global__ void __launch_bounds__(256)
trend_apply_kernel(int64_t n, int64_t n_fit, const double* __restrict__ baseMean, const double* __restrict__ dispGeneEst,
                   const uint8_t* __restrict__ flags, const double* __restrict__ coefs, double* __restrict__ dispFit,
                   double* __restrict__ resid, double* __restrict__ map_start_log, double* __restrict__ log_fit)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flags[i] & CD_FLAG_ALLZERO) { dispFit[i] = NAN; resid[i] = INFINITY; map_start_log[i] = NAN; log_fit[i] = NAN; return; }
    const double* c = coefs + 8 * (i / n_fit);
    const double f = c[0] + c[1] / baseMean[i];
    const double d = dispGeneEst[i];
    dispFit[i] = f;
    resid[i] = (d >= 100.0 * kMinDisp) ? log(d) - log(f) : INFINITY;
    // estimateDispersionsMAP: the search starts at the gene-wise estimate unless that sits more than an order of magnitude
    // below the trend; its prior is centred on the trend.  Both as logarithms, for the line search's refill path.
    const double lf = log_pos(f);
    log_fit[i] = lf;
    map_start_log[i] = (d > 0.1 * f) ? log_pos(d) : lf;
}

cudaError_t launch_trend_apply(int64_t n, int64_t n_fit, const double* baseMean, const double* dispGeneEst, const uint8_t* flags,
                               const double* coefs_dev, double* dispFit, double* resid, double* map_start_log, double* log_fit,
                               cudaStream_t st)
{
    if (n == 0) return cudaSuccess;
    trend_apply_kernel<<<blocks_for(n, 256), 256, 0, st>>>(n, n_fit, baseMean, dispGeneEst, flags, coefs_dev, dispFit, resid,
                                                         map_start_log, log_fit);
    return cudaGetLastError();
}

}  // namespace cd
