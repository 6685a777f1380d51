// context.cu -- the C ABI (include/chicdiff_b200.h) and the orchestration of the hot path:
// DESeq2Wrap's numeric core (chicdiff.R:1540-1674) as a sequence of sm_100a kernels on one
// stream, with the few global steps (size-factor medians, dispersion trend, MAD, theta grid) joined
// across the ranks of a sharded run by all-reduces only: inside the kernels through NVLink peer memory
// where a kernel consumes the sum, by NCCL otherwise.
#include "../../include/chicdiff_b200.h"
#include "kernels.h"
#include "comm.h"
#include "results_host.h"
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <unistd.h>

using namespace cd;

namespace {

thread_local std::string g_create_error;

template <typename T> struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t ensure(size_t count)
    {
        if (count <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) cap = count;
        return e;
    }
};

bool invert_small(const double* A, int p, double* inv)
{
    double a[CD_MAXP][2 * CD_MAXP];
    for (int i = 0; i < p; i++)
        for (int j = 0; j < p; j++) { a[i][j] = A[i * p + j]; a[i][p + j] = (i == j) ? 1.0 : 0.0; }
    for (int k = 0; k < p; k++) {
        int piv = k;
        for (int i = k + 1; i < p; i++) if (fabs(a[i][k]) > fabs(a[piv][k])) piv = i;
        if (fabs(a[piv][k]) < 1e-12) return false;
        if (piv != k) for (int j = 0; j < 2 * p; j++) std::swap(a[k][j], a[piv][j]);
        const double d = a[k][k];
        for (int j = 0; j < 2 * p; j++) a[k][j] /= d;
        for (int i = 0; i < p; i++) if (i != k) {
            const double f = a[i][k];
            if (f != 0.0) for (int j = 0; j < 2 * p; j++) a[i][j] -= f * a[k][j];
        }
    }
    for (int i = 0; i < p; i++) for (int j = 0; j < p; j++) inv[i * p + j] = a[i][p + j];
    return true;
}

bool build_design(int S, int p, const double* X, CdDesign& d)
{
    memset(&d, 0, sizeof(d));
    d.S = S; d.p = p;
    for (int i = 0; i < S * p; i++) d.X[i] = X[i];
    double xtx[CD_MAXP * CD_MAXP], inv[CD_MAXP * CD_MAXP];
    for (int a = 0; a < p; a++)
        for (int b = 0; b < p; b++) {
            double s = 0;
            for (int j = 0; j < S; j++) s += X[j * p + a] * X[j * p + b];
            xtx[a * p + b] = s;
        }
    if (!invert_small(xtx, p, inv)) return false;          // not full rank
    for (int u = 0; u < p; u++)
        for (int j = 0; j < S; j++) {
            double s = 0;
            for (int v = 0; v < p; v++) s += inv[u * p + v] * X[j * p + v];
            d.ls[u * S + j] = s;
        }
    for (int a = 0; a < S; a++)
        for (int b = 0; b < S; b++) {
            double s = 0;
            for (int u = 0; u < p; u++) s += X[a * p + u] * d.ls[u * S + b];
            d.hat[a * S + b] = s;
        }
    d.ncell = 0;
    for (int j = 0; j < S; j++) {
        int found = -1;
        for (int k = 0; k < j && found < 0; k++) {
            bool same = true;
            for (int u = 0; u < p; u++) if (X[j * p + u] != X[k * p + u]) same = false;
            if (same) found = d.cell[k];
        }
        if (found < 0) { found = d.ncell++; d.cell_size[found] = 0; }
        d.cell[j] = found;
        d.cell_size[found]++;
    }
    d.linear_mu = (d.ncell == p);
    d.any3 = 0;
    for (int c = 0; c < d.ncell; c++) if (d.cell_size[c] >= 3) d.any3 = 1;
    return true;
}

double trigamma_host(double x)
{
    double r = 0.0;
    while (x < 10.0) { r += 1.0 / (x * x); x += 1.0; }
    const double f = 1.0 / (x * x);
    return r + 1.0 / x + 0.5 * f +
           (1.0 / x) * f * (1.0 / 6.0 + f * (-1.0 / 30.0 + f * (1.0 / 42.0 + f * (-1.0 / 30.0 +
           f * (5.0 / 66.0 + f * (-691.0 / 2730.0 + f * (7.0 / 6.0)))))));
}

// FP64 peak probe: 8 independent DFMA chains per thread
__global__ void __launch_bounds__(256) dfma_peak_kernel(int iters, double m, double* __restrict__ sink)
{
    double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double c = 1e-9;
#pragma unroll 16
    for (int k = 0; k < iters; k++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456) *sink = r;
}

// line-search evaluations of one fit_disp call: every searched region evaluates the fused posterior once to start and
// once per trip (the count the FP64 roofline of the bench line is built from)
__global__ void count_evals_kernel(int64_t n, const int32_t* __restrict__ iter, unsigned long long* __restrict__ out)
{
    unsigned long long local = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int it = iter[i];
        if (it > 0) local += (unsigned long long)it + 1ull;
    }
    for (int off = 16; off > 0; off >>= 1) local += __shfl_down_sync(0xffffffffu, local, off);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(out, local);
}

__global__ void count_flags_kernel(int64_t n, const uint8_t* __restrict__ flags, unsigned long long* __restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint8_t f = (i < n) ? flags[i] : (uint8_t)CD_FLAG_ALLZERO;
    const unsigned nz = __ballot_sync(0xffffffffu, (i < n) && !(f & CD_FLAG_ALLZERO));
    const unsigned gg = __ballot_sync(0xffffffffu, (i < n) && (f & CD_FLAG_GENE_GRID));
    const unsigned mg = __ballot_sync(0xffffffffu, (i < n) && (f & CD_FLAG_MAP_GRID));
    const unsigned bn = __ballot_sync(0xffffffffu, (i < n) && (f & CD_FLAG_BETA_NOCONV));
    if ((threadIdx.x & 31) == 0) {
        if (nz) atomicAdd(out + 0, (unsigned long long)__popc(nz));
        if (gg) atomicAdd(out + 1, (unsigned long long)__popc(gg));
        if (mg) atomicAdd(out + 2, (unsigned long long)__popc(mg));
        if (bn) atomicAdd(out + 3, (unsigned long long)__popc(bn));
    }
}

// layout of the small device scalar buffer ctx->scal (doubles)
constexpr int kScalSf = 0;            // S size factors
constexpr int kScalXim = 64;          // per fit: moments offset
constexpr int kScalMed = 96;          // per fit: median of the log residuals
constexpr int kScalMad = 128;         // per fit: 1.4826 x median absolute deviation
constexpr int kScalDev = 160;         // per fit: total deviance
constexpr int kScalTrend = 192;       // per fit: 8 doubles (coefficients, status, outer iterations, passes)
constexpr int kScalSums = 384;        // per fit: S + 1 masked column sums of the normalisation factors
constexpr int kScalSize = 1024;
// layout of the pinned host scratch ctx->h_pinned (doubles)
constexpr int kPinTrend = 0, kPinMad = 128, kPinErr = 144, kPinBad = 145, kPinDev = 160, kPinTrendIn = 200, kPinSf = 400;

// layout of the device counter words ctx->counters (unsigned long long; word 11 is free)
constexpr int kCntFlags = 0;          // 4: regions not all zero, gene-wise grid refits, MAP grid refits, GLMs not converged
constexpr int kCntWait = 4;           // 3: SM cycles the trend fit waited for peers' sums, for its own slot, in its first pass
constexpr int kCntBad = 7;            // a double: 1.0 when a count is NA or negative
constexpr int kCntSelBar = 8;         // grid barrier of the medians (unsigned int)
constexpr int kCntTrendBar = 9;       // grid barrier of the trend fit (unsigned int)
constexpr int kCntErr = 10;           // non-zero when a peer-memory exchange gave up
constexpr int kCntFitDispQueue = 12;  // 2: work-queue heads of the line search's two passes
constexpr int kCntPark = 14;          // regions the line search parked
constexpr int kCntWaldQueue = 15;     // work-queue head of the GLM fits
constexpr int kCntSize = 16;

}  // namespace

struct cd_ctx {
    int device = 0;
    cudaStream_t st = nullptr;
    std::string err;
    int64_t launches = 0;
    double timings[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    Comm comm;

    // design
    bool have_design = false;
    CdDesign des{}, des1{};          // user design and the intercept-only design of the theta grid
    DevBuf<CdDesign> des_dev;        // [0] = des, [1] = des1: this context's own device copies (no __constant__ globals)
    // regions / rows
    int64_t n = 0, R = 0;
    bool have_regions = false, have_agg = false, rows_borrowed = false;
    bool have_results = false;       // the arrays of a successful cd_region_test are in device memory
    std::vector<uint8_t> sample_set;
    DevBuf<int64_t> row_off;
    // Per-row columns, double-buffered: cd_set_sample_rows uploads on a copy stream of its own into the buffer the last
    // cd_aggregate did NOT read, so the rows of the next batch cross the bus while the region test of the current
    // one runs (a caller pipelines by setting the next batch's rows between cd_aggregate and cd_region_test).
    DevBuf<int32_t> N_rows, N_rows_alt;
    DevBuf<double> FM_rows, FM_rows_alt;
    cudaStream_t st_copy = nullptr;
    cudaEvent_t ev_copy = nullptr;                 // last upload of the staging round
    cudaEvent_t ev_tab_copy = nullptr, ev_tab_used = nullptr;   // replicate tables: last upload / compute-stream position at upload time
    bool tab_copy_pending = false;
    cudaEvent_t ev_read[2] = {nullptr, nullptr};   // last aggregation kernel that read buffer b
    int front = 0;                                 // buffer the last cd_aggregate consumed
    bool front_used = false;
    std::vector<uint8_t> staged;                   // samples uploaded since then
    int32_t* nbuf(int b) { return b ? N_rows_alt.p : N_rows.p; }
    double* fbuf(int b) { return b ? FM_rows_alt.p : FM_rows.p; }
    int back() const { return front_used ? 1 - front : front; }
    DevBuf<double> BM_rows;          // per-row Bmean, only after cd_assemble(keep_rows)
    bool have_bm_rows = false;
    const int32_t* N_rows_p = nullptr;
    const double* FM_rows_p = nullptr;
    DevBuf<int32_t> K;               // S x n
    DevBuf<double> FM;               // S x n
    DevBuf<int32_t> Kb;              // S x G*n: the counts replicated for the fits of a batch (theta grid)
    int64_t batch_cap = 0;           // virtual regions the work buffers are sized for
    // work buffers (local shard)
    DevBuf<double> nf, mu, baseVar, rough, alpha_init, log_alpha, initial_lp, last_lp, dispMAP, dispersion,
        beta, betaSE, stat, pvalue, deviance, maxCooks;
    DevBuf<int32_t> dispGeneIter, dispIter, betaIter, refit_list;
    // inputs / outputs of the global steps (trend, MAD): local regions only, nothing is gathered
    DevBuf<double> g_baseMean, g_dispGeneEst, g_dispFit, g_resid;
    DevBuf<uint8_t> g_flags;
    DevBuf<double> g_LR;
    DevBuf<unsigned long long> sel_state, sel_hist, sel_aux;
    DevBuf<double> trend_xs;         // scratch of the trend fit: one double per virtual region
    DevBuf<double> start_log, log_fit;   // line-search start values and prior means as logarithms
    DevBuf<double> partial, scal;    // reduction scratch ; device scalars
    DevBuf<unsigned long long> counters;
    DevBuf<unsigned long long> eval_counts;       // per fit_disp call of the last cd_region_test: evaluations
    int n_eval_calls = 0;
    int eval_call_p[16] = {0};                     // design columns of that call
    int64_t eval_call_regions[16] = {0};           // virtual regions of that call
    unsigned long long eval_counts_host[16] = {0};
    double trend_passes_batch = 0;
    double trend_passes = 0;                       // trend passes (= cross-rank rendezvous of the trend fits) of the last region test
    unsigned long long wait_host[3] = {0, 0, 0};
    DevBuf<int32_t> refit_count;
    DevBuf<int64_t> park_row;
    DevBuf<double> park_d;           // 5 x capacity
    DevBuf<int32_t> park_i;          // 2 x capacity
    FitDispPark park{};
    // assembly inputs
    int64_t F = 0;
    int32_t frag_id0 = 0;
    bool have_rmap = false, have_region_rows = false;
    DevBuf<int32_t> frag_chr, frag_start, frag_end, row_bait, row_oe, asm_status;
    std::vector<DevBuf<unsigned char>> tab_blob;
    std::vector<AssembleTables> tabs_host;
    std::vector<uint8_t> tab_set;
    DevBuf<unsigned char> tabs_dev;
    DevBuf<double> avDist;
    // peer-memory all-reduce of the sharded trend fit (set up in cd_comm_init; NCCL path is the fallback)
    bool p2p_ok = false;
    DevBuf<double> p2p_mail;
    DevBuf<double*> p2p_peers_dev;
    std::vector<void*> p2p_opened;
    unsigned long long p2p_epoch = 0;
    bool sel_p2p_ok = false;                      // medians exchange their counters through peer memory too
    DevBuf<unsigned long long> sel_mail;
    DevBuf<unsigned long long*> sel_peers_dev;
    unsigned long long sel_seq = 0;
    // work buffers of cd_results_resident
    DevBuf<unsigned long long> res_key[4], res_small;
    DevBuf<unsigned int> res_idx[2], res_cnt;
    DevBuf<double> res_pv, res_padj, res_bms, res_ps, res_smalld, res_cmin, res_smin;
    DevBuf<unsigned char> res_tmp;
    DevBuf<double> res_in;                               // cd_results_device: uploaded columns
    DevBuf<uint8_t> res_in_flags;
    // columns of the last cd_parse_chinput
    int64_t ch_rows = 0;
    DevBuf<int32_t> ch_bait, ch_oe, ch_N, ch_len;
    DevBuf<double> ch_dist;
    // countput output of the last cd_countput
    int64_t cp_pairs = 0;
    DevBuf<int32_t> cp_bait, cp_oe;
    DevBuf<double> cp_nav, cp_bav, cp_score, cp_mid;
    DevBuf<double> wald_c, wald_b0, wald_b, lfact;
    DevBuf<int32_t> wald_iter;
    WaldScratch wald_ws{};
    double* h_pinned = nullptr;      // pinned host scratch (1024 doubles)
    std::vector<int64_t> shard_n, shard_off;
    int64_t n_tot = 0, g_off = 0;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_user[2] = {nullptr, nullptr};
    // per-section device timing: pairs of events recorded around launches, summed after the final sync
    std::vector<cudaEvent_t> ev_pool;
    std::vector<int> ev_slot;            // section of pair k
    size_t ev_used = 0;
    void tm_begin(int slot)
    {
        if (ev_used + 2 > ev_pool.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a); cudaEventCreate(&b);
            ev_pool.push_back(a); ev_pool.push_back(b);
            ev_slot.push_back(slot);
        }
        ev_slot[ev_used / 2] = slot;
        cudaEventRecord(ev_pool[ev_used], st);
    }
    void tm_end() { cudaEventRecord(ev_pool[ev_used + 1], st); ev_used += 2; }
    void tm_collect()
    {
        for (size_t k = 0; k < ev_used; k += 2) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ev_pool[k], ev_pool[k + 1]) == cudaSuccess) timings[ev_slot[k / 2]] += ms;
        }
        ev_used = 0;
    }

    int fail(int code, const char* fmt, ...)
    {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
};

#define CD_CUDA(ctx, call)                                                                          \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) return (ctx)->fail(CD_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

#define CD_LAUNCHN(ctx, k, call)                                                                    \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        (ctx)->launches += (k);                                                                     \
        if (e_ != cudaSuccess) return (ctx)->fail(CD_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

#define CD_COMM(ctx, call)                                                                          \
    do {                                                                                            \
        std::string m_ = (call);                                                                    \
        if (!m_.empty()) return (ctx)->fail(CD_ECOMM, "%s", m_.c_str());                            \
    } while (0)

extern "C" {

const char* cd_version(void) { return "chicdiff_b200 0.1 (sm_100a)"; }

const char* cd_last_error(const cd_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int cd_create(cd_ctx** out, int device)
{
    if (!out) return CD_EINVAL;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) +
                         " (chicdiff_b200 has no CPU fallback)";
        return CD_ECUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "device ordinal out of range"; return CD_EINVAL; }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return CD_ECUDA; }
    cd_ctx* c = new (std::nothrow) cd_ctx();
    if (!c) return CD_ENOMEM;
    c->device = device;
    if ((e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaMallocHost((void**)&c->h_pinned, 1024 * sizeof(double))) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        delete c;
        return CD_ECUDA;
    }
    cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_tab_copy, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_tab_used, cudaEventDisableTiming);
    for (int k = 0; k < 2; k++) cudaEventCreateWithFlags(&c->ev_read[k], cudaEventDisableTiming);
    for (int k = 0; k < 4; k++) cudaEventCreate(&c->ev[k]);
    for (int k = 0; k < 2; k++) cudaEventCreate(&c->ev_user[k]);
    *out = c;
    return CD_OK;
}

void cd_destroy(cd_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->st);
    if (ctx->st_copy) { cudaStreamSynchronize(ctx->st_copy); cudaStreamDestroy(ctx->st_copy); }
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    if (ctx->ev_tab_copy) cudaEventDestroy(ctx->ev_tab_copy);
    if (ctx->ev_tab_used) cudaEventDestroy(ctx->ev_tab_used);
    for (int k = 0; k < 2; k++) if (ctx->ev_read[k]) cudaEventDestroy(ctx->ev_read[k]);
    for (int k = 0; k < 4; k++) if (ctx->ev[k]) cudaEventDestroy(ctx->ev[k]);
    for (int k = 0; k < 2; k++) if (ctx->ev_user[k]) cudaEventDestroy(ctx->ev_user[k]);
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    for (void* p : ctx->p2p_opened) cudaIpcCloseMemHandle(p);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    cudaStream_t st = ctx->st;
    delete ctx;
    if (st) cudaStreamDestroy(st);
}

int cd_comm_unique_id(cd_ctx* ctx, char id[128])
{
    if (!ctx || !id) return CD_EINVAL;
    CD_COMM(ctx, ctx->comm.unique_id(id));
    return CD_OK;
}

// Exchange cudaIpc handles of two mailboxes per rank so that the trend-fit kernel can all-reduce its sums and the
// median kernel its counters over NVLink themselves.  Every rank runs the SAME sequence of collectives whatever
// happens locally (a failed allocation or handle export is reported in the final agreement all-reduce, never by
// skipping a collective), so no rank can be left waiting in a collective the others do not enter.
static bool open_peer_mailboxes(cd_ctx* ctx, void* mine_ptr, bool local_ok, std::vector<void*>& peers)
{
    const int nr = ctx->comm.nranks, rk = ctx->comm.rank;
    bool ok = local_ok;
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    if (ok && cudaIpcGetMemHandle(&mine, mine_ptr) != cudaSuccess) { cudaGetLastError(); ok = false; }
    // per rank: handle, a validity byte, and -- for peers that live in THIS process (cd_multi: one host thread per GPU) --
    // the process id, the raw device pointer and the device ordinal: such a peer's buffer is mapped by enabling peer
    // access and using the pointer as it is (cudaIpc handles cannot be opened by the process that exported them)
    struct Rec { cudaIpcMemHandle_t h; unsigned char ok; unsigned char pad[7]; long long pid; unsigned long long ptr; int dev; int pad2; };
    const size_t rec = sizeof(Rec);
    DevBuf<unsigned char> hb;
    std::vector<Rec> all((size_t)nr);
    const bool have_buf = hb.ensure((size_t)nr * rec) == cudaSuccess;
    if (have_buf) {
        Rec mine_rec;
        memset(&mine_rec, 0, sizeof(mine_rec));
        mine_rec.h = mine; mine_rec.ok = ok ? 1 : 0; mine_rec.pid = (long long)getpid();
        mine_rec.ptr = (unsigned long long)(uintptr_t)mine_ptr; mine_rec.dev = ctx->device;
        cudaMemcpy(hb.p + (size_t)rk * rec, &mine_rec, rec, cudaMemcpyHostToDevice);
    }
    std::vector<int64_t> counts((size_t)nr, 1), displs((size_t)nr);
    for (int r = 0; r < nr; r++) displs[(size_t)r] = r;
    // (without a staging buffer this rank cannot take part: an allocation of a few hundred bytes failing means the
    //  device is unusable anyway; the collective below would fail on every rank alike)
    if (!have_buf) return false;
    if (!ctx->comm.allgatherv(hb.p + (size_t)rk * rec, hb.p, counts, displs, rec, ctx->st).empty()) ok = false;
    if (cudaMemcpyAsync(all.data(), hb.p, (size_t)nr * rec, cudaMemcpyDeviceToHost, ctx->st) != cudaSuccess) ok = false;
    if (cudaStreamSynchronize(ctx->st) != cudaSuccess) ok = false;
    peers.assign((size_t)nr, nullptr);
    for (int r = 0; r < nr && ok; r++) {
        if (!all[(size_t)r].ok) { ok = false; break; }                                         // that rank could not export
        if (r == rk) { peers[(size_t)r] = mine_ptr; continue; }
        if (all[(size_t)r].pid == (long long)getpid()) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(all[(size_t)r].dev, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = false; break; }
            cudaGetLastError();
            peers[(size_t)r] = (void*)(uintptr_t)all[(size_t)r].ptr;
            continue;
        }
        void* ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, all[(size_t)r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
        ctx->p2p_opened.push_back(ptr);
        peers[(size_t)r] = ptr;
    }
    return ok;
}

// returns an empty string or the reason peer memory is unavailable (identical decision on every rank)
static std::string setup_p2p(cd_ctx* ctx)
{
    ctx->p2p_ok = false;
    ctx->sel_p2p_ok = false;
    for (void* p : ctx->p2p_opened) cudaIpcCloseMemHandle(p);          // a second cd_comm_init starts from scratch
    ctx->p2p_opened.clear();
    const int nr = ctx->comm.nranks;
    if (nr < 2) return "";
    bool local_ok = nr <= 16;                      // median mailbox: 2 x nr x 32 slots of 16 KiB (8 MiB at 8 ranks)
    const char* off = getenv("CHICDIFF_B200_NO_P2P");
    if (off && off[0] == '1') local_ok = false;
    if (local_ok && (ctx->p2p_mail.ensure(trend_p2p_mail_doubles(nr)) != cudaSuccess || ctx->p2p_peers_dev.ensure((size_t)nr) != cudaSuccess ||
                     ctx->sel_mail.ensure(sel_p2p_mail_words(nr)) != cudaSuccess || ctx->sel_peers_dev.ensure((size_t)nr) != cudaSuccess))
        local_ok = false;
    if (local_ok) {
        cudaMemset(ctx->p2p_mail.p, 0, sizeof(double) * trend_p2p_mail_doubles(nr));
        cudaMemset(ctx->sel_mail.p, 0, sizeof(unsigned long long) * sel_p2p_mail_words(nr));
    }
    std::vector<void*> peers, sel_peers;
    const bool ok = open_peer_mailboxes(ctx, ctx->p2p_mail.p, local_ok, peers);
    const bool sel_ok = open_peer_mailboxes(ctx, ctx->sel_mail.p, local_ok, sel_peers);
    // every rank must agree, otherwise one would wait in a kernel for a peer that never writes its mailbox
    double flag[2] = {ok ? 0.0 : 1.0, sel_ok ? 0.0 : 1.0};
    DevBuf<double> fb;
    if (fb.ensure(2) != cudaSuccess) return "cudaMalloc failed";
    cudaMemcpy(fb.p, flag, sizeof(flag), cudaMemcpyHostToDevice);
    const std::string e = ctx->comm.allreduce_sum(fb.p, 2, ctx->st);
    if (!e.empty()) return e;
    cudaMemcpyAsync(flag, fb.p, sizeof(flag), cudaMemcpyDeviceToHost, ctx->st);
    cudaStreamSynchronize(ctx->st);
    if (flag[0] != 0.0 || flag[1] != 0.0)
        return "peer memory between the GPUs of this run is unavailable on at least one rank (cudaIpc / NVLink peer access; more "
               "than 16 ranks; or CHICDIFF_B200_NO_P2P=1): the global steps of a sharded run exchange their sums inside the kernels";
    cudaMemcpy(ctx->p2p_peers_dev.p, peers.data(), sizeof(double*) * (size_t)nr, cudaMemcpyHostToDevice);
    cudaMemcpy(ctx->sel_peers_dev.p, sel_peers.data(), sizeof(void*) * (size_t)nr, cudaMemcpyHostToDevice);
    ctx->p2p_ok = true;
    ctx->sel_p2p_ok = true;
    return "";
}

int cd_comm_init(cd_ctx* ctx, int nranks, int rank, const char id[128])
{
    if (!ctx || !id) return CD_EINVAL;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_COMM(ctx, ctx->comm.init(nranks, rank, id));
    if (!ctx->counters.p) {
        CD_CUDA(ctx, ctx->counters.ensure(kCntSize));
        CD_CUDA(ctx, cudaMemset(ctx->counters.p, 0, kCntSize * sizeof(unsigned long long)));
    }
    const std::string why = setup_p2p(ctx);
    if (!why.empty()) {
        // fall back to a single-rank context rather than leaving a communicator nobody can use
        ctx->comm.init(1, 0, id);
        return ctx->fail(CD_ECOMM, "cd_comm_init: %s", why.c_str());
    }
    return CD_OK;
}

int cd_comm_info(const cd_ctx* ctx, int* nranks, int* rank, int* peer_memory_allreduce)
{
    if (!ctx) return CD_EINVAL;
    if (nranks) *nranks = ctx->comm.nranks;
    if (rank) *rank = ctx->comm.rank;
    if (peer_memory_allreduce) *peer_memory_allreduce = (ctx->p2p_ok ? 1 : 0) | (ctx->sel_p2p_ok ? 2 : 0);
    return CD_OK;
}

int cd_plan_shards(int64_t n, const int32_t* region_bait, const int64_t* row_off, int nshards, int64_t* bounds)
{
    if (n < 0 || nshards < 1 || !bounds || (n > 0 && (!region_bait || !row_off))) return CD_EINVAL;
    bounds[0] = 0;
    const int64_t total = n > 0 ? row_off[n] - row_off[0] : 0;
    int64_t i = 0;
    for (int k = 1; k < nshards; k++) {
        const int64_t target = row_off ? row_off[0] + (total * k) / nshards : 0;
        // first region whose rows start at or after the target ...
        int64_t lo = i, hi = n;
        while (lo < hi) {
            const int64_t mid = (lo + hi) / 2;
            if (row_off[mid] < target) lo = mid + 1; else hi = mid;
        }
        i = lo;
        // ... moved forward to the next bait boundary
        while (i > 0 && i < n && region_bait[i] == region_bait[i - 1]) i++;
        bounds[k] = i;
    }
    bounds[nshards] = n;
    for (int k = 1; k <= nshards; k++) if (bounds[k] < bounds[k - 1]) bounds[k] = bounds[k - 1];
    return CD_OK;
}

int cd_set_design(cd_ctx* ctx, int S, int p, const double* X)
{
    if (!ctx) return CD_EINVAL;
    if (!X || S < 2 || S > CD_MAXS || p < 1 || p > CD_MAXP)
        return ctx->fail(CD_EINVAL, "cd_set_design: need 2 <= S <= %d and 1 <= p <= %d", CD_MAXS, CD_MAXP);
    if (S <= p) return ctx->fail(CD_EINVAL, "cd_set_design: S <= p: no residual degrees of freedom (DESeq2 stops here too)");
    if (!build_design(S, p, X, ctx->des)) return ctx->fail(CD_EINVAL, "cd_set_design: the model matrix is not full rank");
    double ones[CD_MAXS];
    for (int j = 0; j < S; j++) ones[j] = 1.0;
    build_design(S, 1, ones, ctx->des1);
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->des_dev.ensure(2));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->des_dev.p, &ctx->des, sizeof(CdDesign), cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->des_dev.p + 1, &ctx->des1, sizeof(CdDesign), cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));          // the sources are members, but be explicit about lifetime
    ctx->have_design = true;
    ctx->have_regions = ctx->have_agg = false;
    ctx->sample_set.assign((size_t)S, 0);
    ctx->staged.assign((size_t)S, 0);
    ctx->front_used = false;
    return CD_OK;
}

int cd_set_regions(cd_ctx* ctx, int64_t n, const int64_t* row_off)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_design) return ctx->fail(CD_EINVAL, "cd_set_regions: call cd_set_design first");
    if (n < 0 || n > 2000000000LL || !row_off) return ctx->fail(CD_EINVAL, "cd_set_regions: bad n / row_off");
    for (int64_t i = 0; i < n; i++)
        if (row_off[i + 1] < row_off[i]) return ctx->fail(CD_EINVAL, "cd_set_regions: row_off must be non-decreasing");
    if (row_off[0] != 0) return ctx->fail(CD_EINVAL, "cd_set_regions: row_off[0] must be 0");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->row_off.ensure((size_t)n + 1));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->row_off.p, row_off, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    ctx->n = n;
    ctx->R = row_off[n];
    ctx->have_regions = true;
    ctx->have_bm_rows = false;
    ctx->have_region_rows = false;
    ctx->have_agg = false;
    ctx->rows_borrowed = false;
    ctx->N_rows_p = nullptr; ctx->FM_rows_p = nullptr;
    std::fill(ctx->sample_set.begin(), ctx->sample_set.end(), 0);
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st_copy));
    std::fill(ctx->staged.begin(), ctx->staged.end(), 0);
    ctx->front_used = false;
    return CD_OK;
}

int cd_set_sample_rows(cd_ctx* ctx, int s, int64_t R, const int32_t* N, const double* fullmean)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions) return ctx->fail(CD_EINVAL, "cd_set_sample_rows: call cd_set_regions first");
    const int S = ctx->des.S;
    if (s < 0 || s >= S || R != ctx->R || (R > 0 && (!N || !fullmean)))
        return ctx->fail(CD_EINVAL, "cd_set_sample_rows: sample index or row count does not match the regions");
    if (ctx->rows_borrowed) return ctx->fail(CD_EINVAL, "cd_set_sample_rows: rows were set with cd_set_rows_device");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const int b = ctx->back();
    if (b == 0) { CD_CUDA(ctx, ctx->N_rows.ensure((size_t)S * (size_t)R)); CD_CUDA(ctx, ctx->FM_rows.ensure((size_t)S * (size_t)R)); }
    else { CD_CUDA(ctx, ctx->N_rows_alt.ensure((size_t)S * (size_t)R)); CD_CUDA(ctx, ctx->FM_rows_alt.ensure((size_t)S * (size_t)R)); }
    bool first_of_round = true;
    for (uint8_t f : ctx->staged) if (f) first_of_round = false;
    // the buffer being filled was read by the aggregation two batches ago: that kernel must be done
    if (first_of_round) CD_CUDA(ctx, cudaStreamWaitEvent(ctx->st_copy, ctx->ev_read[b], 0));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->nbuf(b) + (size_t)s * R, N, sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, ctx->st_copy));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->fbuf(b) + (size_t)s * R, fullmean, sizeof(double) * (size_t)R, cudaMemcpyHostToDevice, ctx->st_copy));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev_copy, ctx->st_copy));
    ctx->staged[(size_t)s] = 1;
    ctx->sample_set[(size_t)s] = 1;
    // (the matrices of the last cd_aggregate stay valid: these rows belong to the NEXT cd_aggregate, and a region test of
    //  the current batch may run while they are on their way)
    return CD_OK;            // asynchronous: the host buffers must stay valid until the next cd_aggregate has returned
}

int cd_set_rows_device(cd_ctx* ctx, int64_t R, const int32_t* N_dev, const double* fullmean_dev)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions) return ctx->fail(CD_EINVAL, "cd_set_rows_device: call cd_set_regions first");
    if (R != ctx->R || (R > 0 && (!N_dev || !fullmean_dev))) return ctx->fail(CD_EINVAL, "cd_set_rows_device: row count mismatch");
    ctx->N_rows_p = N_dev; ctx->FM_rows_p = fullmean_dev;
    ctx->rows_borrowed = true;
    std::fill(ctx->sample_set.begin(), ctx->sample_set.end(), 1);
    ctx->have_agg = false;
    return CD_OK;
}

int cd_set_aggregated(cd_ctx* ctx, int64_t n, const int32_t* K, const double* fullmean)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_design) return ctx->fail(CD_EINVAL, "cd_set_aggregated: call cd_set_design first");
    if (n < 0 || (n > 0 && (!K || !fullmean))) return ctx->fail(CD_EINVAL, "cd_set_aggregated: bad arguments");
    const int S = ctx->des.S;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->K.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, ctx->FM.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->K.p, K, sizeof(int32_t) * (size_t)S * (size_t)n, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->FM.p, fullmean, sizeof(double) * (size_t)S * (size_t)n, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    ctx->n = n;
    ctx->have_agg = true;
    return CD_OK;
}

int cd_set_rmap(cd_ctx* ctx, int64_t F, int32_t frag_id0, const int32_t* chr, const int32_t* start, const int32_t* end)
{
    if (!ctx) return CD_EINVAL;
    if (F < 1 || !chr || !start || !end) return ctx->fail(CD_EINVAL, "cd_set_rmap: bad arguments");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->frag_chr.ensure((size_t)F)); CD_CUDA(ctx, ctx->frag_start.ensure((size_t)F)); CD_CUDA(ctx, ctx->frag_end.ensure((size_t)F));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->frag_chr.p, chr, sizeof(int32_t) * (size_t)F, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->frag_start.p, start, sizeof(int32_t) * (size_t)F, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->frag_end.p, end, sizeof(int32_t) * (size_t)F, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    ctx->F = F; ctx->frag_id0 = frag_id0; ctx->have_rmap = true;
    return CD_OK;
}

int cd_region_universe(cd_ctx* ctx, int64_t m, const int32_t* peak_bait, const int32_t* peak_oe, int ru_expand, int64_t* R_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_design || !ctx->have_rmap) return ctx->fail(CD_EINVAL, "cd_region_universe: call cd_set_design and cd_set_rmap first");
    if (m < 0 || m > 2000000000LL || ru_expand < 1 || (m > 0 && (!peak_bait || !peak_oe)))
        return ctx->fail(CD_EINVAL, "cd_region_universe: bad arguments (RUexpand must be >= 1)");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    DevBuf<int32_t> pb, po;
    DevBuf<int64_t> counts;
    DevBuf<unsigned char> tmp;
    CD_CUDA(ctx, pb.ensure((size_t)m)); CD_CUDA(ctx, po.ensure((size_t)m)); CD_CUDA(ctx, counts.ensure((size_t)m + 1));
    CD_CUDA(ctx, ctx->row_off.ensure((size_t)m + 1));
    CD_CUDA(ctx, ctx->asm_status.ensure(1));
    CD_CUDA(ctx, cudaMemcpyAsync(pb.p, peak_bait, sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice, st));
    CD_CUDA(ctx, cudaMemcpyAsync(po.p, peak_oe, sizeof(int32_t) * (size_t)m, cudaMemcpyHostToDevice, st));
    CD_CUDA(ctx, cudaMemsetAsync(counts.p, 0, sizeof(int64_t) * ((size_t)m + 1), st));
    CD_CUDA(ctx, cudaMemsetAsync(ctx->asm_status.p, 0, sizeof(int32_t), st));
    CD_LAUNCHN(ctx, 1, ru_launch_count(m, pb.p, po.p, ru_expand, ctx->F, ctx->frag_id0, ctx->frag_chr.p, counts.p, ctx->asm_status.p, st));
    size_t bytes = 0;
    CD_CUDA(ctx, ru_launch_scan(m, counts.p, ctx->row_off.p, nullptr, bytes, st));
    CD_CUDA(ctx, tmp.ensure(bytes));
    CD_CUDA(ctx, ru_launch_scan(m, counts.p, ctx->row_off.p, tmp.p, bytes, st));
    int64_t R = 0;
    int32_t status = 0;
    CD_CUDA(ctx, cudaMemcpyAsync(&R, ctx->row_off.p + m, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(&status, ctx->asm_status.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    if (status & 1) return ctx->fail(CD_EINVAL, "Invalid parameters: a peak has oeID == baitID (.expandAvoidBait stops here too)");
    if (status & 2) return ctx->fail(CD_EINVAL, "cd_region_universe: a baitID is not in the rmap");
    CD_CUDA(ctx, ctx->row_bait.ensure((size_t)R)); CD_CUDA(ctx, ctx->row_oe.ensure((size_t)R));
    CD_LAUNCHN(ctx, 1, ru_launch_fill(m, pb.p, po.p, ru_expand, ctx->F, ctx->frag_id0, ctx->frag_chr.p, ctx->row_off.p,
                                      ctx->row_bait.p, ctx->row_oe.p, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->n = m; ctx->R = R;
    ctx->have_regions = true; ctx->have_region_rows = true; ctx->have_agg = false; ctx->rows_borrowed = false;
    ctx->N_rows_p = nullptr; ctx->FM_rows_p = nullptr;
    std::fill(ctx->sample_set.begin(), ctx->sample_set.end(), 0);
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st_copy));
    std::fill(ctx->staged.begin(), ctx->staged.end(), 0);
    ctx->front_used = false;
    if (R_out) *R_out = R;
    return CD_OK;
}

int cd_get_region_universe(cd_ctx* ctx, int64_t* row_off_out, int32_t* row_bait_out, int32_t* row_oe_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions || !ctx->have_region_rows) return ctx->fail(CD_EINVAL, "cd_get_region_universe: no region universe on the device");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    if (row_off_out) CD_CUDA(ctx, cudaMemcpyAsync(row_off_out, ctx->row_off.p, sizeof(int64_t) * ((size_t)ctx->n + 1), cudaMemcpyDeviceToHost, ctx->st));
    if (row_bait_out) CD_CUDA(ctx, cudaMemcpyAsync(row_bait_out, ctx->row_bait.p, sizeof(int32_t) * (size_t)ctx->R, cudaMemcpyDeviceToHost, ctx->st));
    if (row_oe_out) CD_CUDA(ctx, cudaMemcpyAsync(row_oe_out, ctx->row_oe.p, sizeof(int32_t) * (size_t)ctx->R, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    return CD_OK;
}

int cd_parse_chinput(cd_ctx* ctx, const char* text, int64_t nbytes, int64_t* n_rows_out)
{
    if (!ctx) return CD_EINVAL;
    if (nbytes < 0 || nbytes > 2147483647LL || (nbytes > 0 && !text)) return ctx->fail(CD_EINVAL, "cd_parse_chinput: bad arguments (at most 2^31-1 bytes per call)");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    ctx->ch_rows = 0;
    if (n_rows_out) *n_rows_out = 0;
    if (nbytes == 0) return CD_OK;
    DevBuf<char> d_text;
    DevBuf<uint8_t> flag, valid;
    DevBuf<int64_t> starts, d_count;
    DevBuf<unsigned char> tmp;
    DevBuf<int32_t> t_bait, t_oe, t_N, t_len;
    DevBuf<double> t_dist;
    CD_CUDA(ctx, d_text.ensure((size_t)nbytes)); CD_CUDA(ctx, flag.ensure((size_t)nbytes)); CD_CUDA(ctx, d_count.ensure(1));
    CD_CUDA(ctx, cudaMemcpyAsync(d_text.p, text, (size_t)nbytes, cudaMemcpyHostToDevice, st));
    CD_LAUNCHN(ctx, 1, ch_launch_line_flags(nbytes, d_text.p, flag.p, st));
    // every byte could start a line (runs of blank lines), so the offset array is sized for that
    size_t bytes = 0;
    CD_CUDA(ctx, starts.ensure((size_t)nbytes));
    {
        int64_t nl = 0;
        CD_CUDA(ctx, ch_line_starts(nullptr, bytes, flag.p, starts.p, d_count.p, nbytes, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        CD_CUDA(ctx, ch_line_starts(tmp.p, bytes, flag.p, starts.p, d_count.p, nbytes, st));
        CD_CUDA(ctx, cudaMemcpyAsync(&nl, d_count.p, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaStreamSynchronize(st));
        const size_t L = (size_t)nl;
        CD_CUDA(ctx, t_bait.ensure(L)); CD_CUDA(ctx, t_oe.ensure(L)); CD_CUDA(ctx, t_N.ensure(L)); CD_CUDA(ctx, t_len.ensure(L));
        CD_CUDA(ctx, t_dist.ensure(L)); CD_CUDA(ctx, valid.ensure(L));
        CD_LAUNCHN(ctx, 1, ch_launch_parse(nl, nbytes, d_text.p, starts.p, t_bait.p, t_oe.p, t_N.p, t_len.p, t_dist.p, valid.p, st));
        CD_CUDA(ctx, ctx->ch_bait.ensure(L)); CD_CUDA(ctx, ctx->ch_oe.ensure(L)); CD_CUDA(ctx, ctx->ch_N.ensure(L));
        CD_CUDA(ctx, ctx->ch_len.ensure(L)); CD_CUDA(ctx, ctx->ch_dist.ensure(L));
        bytes = 0;
        CD_CUDA(ctx, ch_compact_f64(nullptr, bytes, t_dist.p, valid.p, ctx->ch_dist.p, d_count.p, nl, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        size_t b2 = bytes;
        CD_CUDA(ctx, ch_compact_f64(tmp.p, b2, t_dist.p, valid.p, ctx->ch_dist.p, d_count.p, nl, st));
        b2 = bytes; CD_CUDA(ctx, ch_compact_i32(tmp.p, b2, t_bait.p, valid.p, ctx->ch_bait.p, d_count.p, nl, st));
        b2 = bytes; CD_CUDA(ctx, ch_compact_i32(tmp.p, b2, t_oe.p, valid.p, ctx->ch_oe.p, d_count.p, nl, st));
        b2 = bytes; CD_CUDA(ctx, ch_compact_i32(tmp.p, b2, t_N.p, valid.p, ctx->ch_N.p, d_count.p, nl, st));
        b2 = bytes; CD_CUDA(ctx, ch_compact_i32(tmp.p, b2, t_len.p, valid.p, ctx->ch_len.p, d_count.p, nl, st));
        int64_t rows = 0;
        CD_CUDA(ctx, cudaMemcpyAsync(&rows, d_count.p, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaStreamSynchronize(st));
        ctx->ch_rows = rows;
        if (n_rows_out) *n_rows_out = rows;
    }
    return CD_OK;
}

int cd_get_chinput(cd_ctx* ctx, int32_t* baitID, int32_t* otherEndID, int32_t* N, int32_t* otherEndLen, double* distSign)
{
    if (!ctx) return CD_EINVAL;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t m = (size_t)ctx->ch_rows;
    if (!m) return CD_OK;
    cudaStream_t st = ctx->st;
    if (baitID) CD_CUDA(ctx, cudaMemcpyAsync(baitID, ctx->ch_bait.p, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, st));
    if (otherEndID) CD_CUDA(ctx, cudaMemcpyAsync(otherEndID, ctx->ch_oe.p, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, st));
    if (N) CD_CUDA(ctx, cudaMemcpyAsync(N, ctx->ch_N.p, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, st));
    if (otherEndLen) CD_CUDA(ctx, cudaMemcpyAsync(otherEndLen, ctx->ch_len.p, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, st));
    if (distSign) CD_CUDA(ctx, cudaMemcpyAsync(distSign, ctx->ch_dist.p, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    return CD_OK;
}

int cd_countput(cd_ctx* ctx, int n_reps, const cd_chicago_rows* reps, int64_t* n_pairs_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_rmap) return ctx->fail(CD_EINVAL, "cd_countput: call cd_set_rmap first");
    if (n_reps < 1 || !reps) return ctx->fail(CD_EINVAL, "cd_countput: bad arguments");
    int64_t T = 0;
    for (int r = 0; r < n_reps; r++) {
        if (reps[r].rows < 0 || (reps[r].rows > 0 && (!reps[r].baitID || !reps[r].otherEndID || !reps[r].N || !reps[r].Bmean || !reps[r].score)))
            return ctx->fail(CD_EINVAL, "cd_countput: replicate %d has null columns", r);
        T += reps[r].rows;
    }
    if (T > 4000000000LL) return ctx->fail(CD_EINVAL, "cd_countput: more than 4e9 rows in one condition");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    DevBuf<int32_t> bait, oe, N;
    DevBuf<double> Bm, sc, g_nav, g_bav, g_score;
    DevBuf<unsigned long long> k0, k1, g_key;
    DevBuf<unsigned int> i0, i1, g_first, g_first_sorted, ord0, ord1;
    DevBuf<int64_t> head, slot;
    DevBuf<unsigned char> tmp;
    const size_t Ts = (size_t)T;
    CD_CUDA(ctx, bait.ensure(Ts)); CD_CUDA(ctx, oe.ensure(Ts)); CD_CUDA(ctx, N.ensure(Ts)); CD_CUDA(ctx, Bm.ensure(Ts)); CD_CUDA(ctx, sc.ensure(Ts));
    CD_CUDA(ctx, k0.ensure(Ts)); CD_CUDA(ctx, k1.ensure(Ts)); CD_CUDA(ctx, i0.ensure(Ts)); CD_CUDA(ctx, i1.ensure(Ts));
    CD_CUDA(ctx, head.ensure(Ts + 1)); CD_CUDA(ctx, slot.ensure(Ts + 1));
    int64_t base = 0;
    for (int r = 0; r < n_reps; r++) {
        const size_t m = (size_t)reps[r].rows;
        if (!m) continue;
        CD_CUDA(ctx, cudaMemcpyAsync(bait.p + base, reps[r].baitID, sizeof(int32_t) * m, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(oe.p + base, reps[r].otherEndID, sizeof(int32_t) * m, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(N.p + base, reps[r].N, sizeof(int32_t) * m, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(Bm.p + base, reps[r].Bmean, sizeof(double) * m, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(sc.p + base, reps[r].score, sizeof(double) * m, cudaMemcpyHostToDevice, st));
        CD_LAUNCHN(ctx, 1, cp_launch_keys(reps[r].rows, base, bait.p + base, oe.p + base, k0.p, i0.p, st));
        base += reps[r].rows;
    }
    int64_t G = 0;
    if (T > 0) {
        size_t bytes = 0;
        CD_CUDA(ctx, cp_sort_pairs_u64(nullptr, bytes, k0.p, k1.p, i0.p, i1.p, T, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        CD_CUDA(ctx, cp_sort_pairs_u64(tmp.p, bytes, k0.p, k1.p, i0.p, i1.p, T, st));
        CD_LAUNCHN(ctx, 1, cp_launch_heads(T, k1.p, head.p, st));
        CD_CUDA(ctx, cudaMemsetAsync(head.p + T, 0, sizeof(int64_t), st));
        bytes = 0;
        CD_CUDA(ctx, cp_scan_i64(nullptr, bytes, head.p, slot.p, T + 1, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        CD_CUDA(ctx, cp_scan_i64(tmp.p, bytes, head.p, slot.p, T + 1, st));
        CD_CUDA(ctx, cudaMemcpyAsync(&G, slot.p + T, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaStreamSynchronize(st));
        const size_t Gs = (size_t)G;
        CD_CUDA(ctx, g_key.ensure(Gs)); CD_CUDA(ctx, g_nav.ensure(Gs)); CD_CUDA(ctx, g_bav.ensure(Gs)); CD_CUDA(ctx, g_score.ensure(Gs));
        CD_CUDA(ctx, g_first.ensure(Gs)); CD_CUDA(ctx, g_first_sorted.ensure(Gs)); CD_CUDA(ctx, ord0.ensure(Gs)); CD_CUDA(ctx, ord1.ensure(Gs));
        CD_LAUNCHN(ctx, 1, cp_launch_reduce(T, k1.p, i1.p, head.p, slot.p, N.p, Bm.p, sc.p, g_key.p, g_nav.p, g_bav.p, g_score.p, g_first.p, st));
        CD_LAUNCHN(ctx, 1, cp_launch_iota(G, ord0.p, st));
        bytes = 0;
        CD_CUDA(ctx, cp_sort_pairs_u32(nullptr, bytes, g_first.p, g_first_sorted.p, ord0.p, ord1.p, G, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        CD_CUDA(ctx, cp_sort_pairs_u32(tmp.p, bytes, g_first.p, g_first_sorted.p, ord0.p, ord1.p, G, st));
        CD_CUDA(ctx, ctx->cp_bait.ensure(Gs)); CD_CUDA(ctx, ctx->cp_oe.ensure(Gs)); CD_CUDA(ctx, ctx->cp_nav.ensure(Gs));
        CD_CUDA(ctx, ctx->cp_bav.ensure(Gs)); CD_CUDA(ctx, ctx->cp_score.ensure(Gs)); CD_CUDA(ctx, ctx->cp_mid.ensure(Gs));
        CD_LAUNCHN(ctx, 1, cp_launch_gather(G, ord1.p, g_key.p, g_nav.p, g_bav.p, g_score.p, ctx->F, ctx->frag_id0, ctx->frag_start.p,
                                            ctx->frag_end.p, ctx->cp_bait.p, ctx->cp_oe.p, ctx->cp_nav.p, ctx->cp_bav.p, ctx->cp_score.p,
                                            ctx->cp_mid.p, st));
        CD_CUDA(ctx, cudaStreamSynchronize(st));
    }
    ctx->cp_pairs = G;
    if (n_pairs_out) *n_pairs_out = G;
    return CD_OK;
}

int cd_get_countput(cd_ctx* ctx, int32_t* baitID, int32_t* otherEndID, double* Nav, double* Bav, double* score, double* oeID_mid)
{
    if (!ctx) return CD_EINVAL;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t G = (size_t)ctx->cp_pairs;
    if (G == 0) return CD_OK;
    cudaStream_t st = ctx->st;
    if (baitID) CD_CUDA(ctx, cudaMemcpyAsync(baitID, ctx->cp_bait.p, sizeof(int32_t) * G, cudaMemcpyDeviceToHost, st));
    if (otherEndID) CD_CUDA(ctx, cudaMemcpyAsync(otherEndID, ctx->cp_oe.p, sizeof(int32_t) * G, cudaMemcpyDeviceToHost, st));
    if (Nav) CD_CUDA(ctx, cudaMemcpyAsync(Nav, ctx->cp_nav.p, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    if (Bav) CD_CUDA(ctx, cudaMemcpyAsync(Bav, ctx->cp_bav.p, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    if (score) CD_CUDA(ctx, cudaMemcpyAsync(score, ctx->cp_score.p, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    if (oeID_mid) CD_CUDA(ctx, cudaMemcpyAsync(oeID_mid, ctx->cp_mid.p, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    return CD_OK;
}

int cd_set_region_rows(cd_ctx* ctx, int64_t R, const int32_t* row_bait, const int32_t* row_oe)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions) return ctx->fail(CD_EINVAL, "cd_set_region_rows: call cd_set_regions first");
    if (R != ctx->R || (R > 0 && (!row_bait || !row_oe))) return ctx->fail(CD_EINVAL, "cd_set_region_rows: row count does not match the regions");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->row_bait.ensure((size_t)R)); CD_CUDA(ctx, ctx->row_oe.ensure((size_t)R));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->row_bait.p, row_bait, sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->row_oe.p, row_oe, sizeof(int32_t) * (size_t)R, cudaMemcpyHostToDevice, ctx->st));
    ctx->have_region_rows = true;
    ctx->have_agg = false;
    return CD_OK;
}

int cd_set_sample_tables(cd_ctx* ctx, int s, const cd_sample_tables* t)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_design || !ctx->have_rmap) return ctx->fail(CD_EINVAL, "cd_set_sample_tables: call cd_set_design and cd_set_rmap first");
    const int S = ctx->des.S;
    if (s < 0 || s >= S || !t || !t->s_j || !t->tblb || !t->s_i || !t->tlb || !t->tmean || !t->cnt_off || t->n_tblb < 1 || t->n_tlb < 1)
        return ctx->fail(CD_EINVAL, "cd_set_sample_tables: bad arguments");
    const int64_t F = ctx->F;
    const int64_t ncnt = t->cnt_off[F];
    if (t->cnt_off[0] != 0 || ncnt < 0 || (ncnt > 0 && (!t->cnt_oe || !t->cnt_N))) return ctx->fail(CD_EINVAL, "cd_set_sample_tables: bad count table");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    if ((int)ctx->tab_blob.size() != S) { ctx->tab_blob.clear(); ctx->tab_blob.resize((size_t)S); ctx->tabs_host.assign((size_t)S, AssembleTables{}); ctx->tab_set.assign((size_t)S, 0); }
    // one device allocation per replicate, 256-byte aligned sections
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t nt = (size_t)t->n_tblb * (size_t)t->n_tlb;
    size_t off[11], pos = 0;
    const size_t sizes[10] = {sizeof(double) * (size_t)F, sizeof(int32_t) * (size_t)F, sizeof(double) * (size_t)F, sizeof(int32_t) * (size_t)F,
                              sizeof(double) * nt, sizeof(double) * (size_t)t->n_tblb, sizeof(double) * 10, sizeof(int64_t) * ((size_t)F + 1),
                              sizeof(int32_t) * (size_t)ncnt, sizeof(int32_t) * (size_t)ncnt};
    for (int k = 0; k < 10; k++) { off[k] = pos; pos += al(sizes[k]); }
    off[10] = pos;
    DevBuf<unsigned char>& blob = ctx->tab_blob[(size_t)s];
    CD_CUDA(ctx, blob.ensure(pos));
    // The copies run on the context's copy stream, like the region rows': cd_assemble is the only reader of these tables
    // and returns only when its kernel is done, so the tables of the NEXT batch can cross the bus while the region test
    // of the current one runs.  (Ordered after anything the compute stream still does with this blob:
    // cd_build_sample_tables, cd_get_sample_tables.)
    CD_CUDA(ctx, cudaEventRecord(ctx->ev_tab_used, ctx->st));
    CD_CUDA(ctx, cudaStreamWaitEvent(ctx->st_copy, ctx->ev_tab_used, 0));
    const void* src[10] = {t->s_j, t->tblb, t->s_i, t->tlb, t->tmean, nullptr, t->distfun, t->cnt_off, t->cnt_oe, t->cnt_N};
    for (int k = 0; k < 10; k++)
        if (src[k] && sizes[k]) CD_CUDA(ctx, cudaMemcpyAsync(blob.p + off[k], src[k], sizes[k], cudaMemcpyHostToDevice, ctx->st_copy));
    AssembleTables& a = ctx->tabs_host[(size_t)s];
    a.s_j = (const double*)(blob.p + off[0]); a.tblb = (const int32_t*)(blob.p + off[1]);
    a.s_i = (const double*)(blob.p + off[2]); a.tlb = (const int32_t*)(blob.p + off[3]);
    a.tmean = (const double*)(blob.p + off[4]); a.tmin = (const double*)(blob.p + off[5]);
    a.distfun = (const double*)(blob.p + off[6]); a.cnt_off = (const int64_t*)(blob.p + off[7]);
    a.cnt_oe = (const int32_t*)(blob.p + off[8]); a.cnt_N = (const int32_t*)(blob.p + off[9]);
    a.n_tblb = t->n_tblb; a.n_tlb = t->n_tlb;
    CD_LAUNCHN(ctx, 1, launch_tmin(t->n_tblb, t->n_tlb, a.tmean, (double*)(blob.p + off[5]), ctx->st_copy));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev_tab_copy, ctx->st_copy));
    ctx->tab_copy_pending = true;
    ctx->tab_set[(size_t)s] = 1;
    // (the matrices of the last cd_assemble stay valid: these tables belong to the NEXT one)
    return CD_OK;           // asynchronous: the host arrays must stay valid until the next cd_assemble has returned
}

int cd_build_sample_tables(cd_ctx* ctx, int s, const cd_chicago_table* t)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_design || !ctx->have_rmap) return ctx->fail(CD_EINVAL, "cd_build_sample_tables: call cd_set_design and cd_set_rmap first");
    const int S = ctx->des.S;
    if (s < 0 || s >= S || !t || t->rows < 0 || t->rows > 4000000000LL || t->n_tblb < 1 || t->n_tlb < 1 || t->cnt_rows < 0 || t->cnt_rows > 4000000000LL)
        return ctx->fail(CD_EINVAL, "cd_build_sample_tables: bad arguments");
    const int64_t m = t->rows;
    if (m > 0 && (!t->baitID || !t->otherEndID || !t->s_j || !t->s_i || !t->tblb || !t->tlb || !t->Tmean))
        return ctx->fail(CD_EINVAL, "cd_build_sample_tables: null column");
    const bool own_counts = t->cnt_rows == 0;
    if (own_counts && m > 0 && !t->N) return ctx->fail(CD_EINVAL, "cd_build_sample_tables: neither count rows nor the table's N column given");
    if (ctx->tab_copy_pending) { cudaStreamWaitEvent(ctx->st, ctx->ev_tab_copy, 0); ctx->tab_copy_pending = false; }
    if (!own_counts && (!t->cnt_baitID || !t->cnt_otherEndID || !t->cnt_N)) return ctx->fail(CD_EINVAL, "cd_build_sample_tables: null count column");
    const int64_t mc = own_counts ? m : t->cnt_rows;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    const int64_t F = ctx->F;
    if ((int)ctx->tab_blob.size() != S) { ctx->tab_blob.clear(); ctx->tab_blob.resize((size_t)S); ctx->tabs_host.assign((size_t)S, AssembleTables{}); ctx->tab_set.assign((size_t)S, 0); }
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t nt = (size_t)t->n_tblb * (size_t)t->n_tlb;
    size_t off[11], pos = 0;
    const size_t sizes[10] = {sizeof(double) * (size_t)F, sizeof(int32_t) * (size_t)F, sizeof(double) * (size_t)F, sizeof(int32_t) * (size_t)F,
                              sizeof(double) * nt, sizeof(double) * (size_t)t->n_tblb, sizeof(double) * 10, sizeof(int64_t) * ((size_t)F + 1),
                              sizeof(int32_t) * (size_t)mc, sizeof(int32_t) * (size_t)mc};
    for (int k = 0; k < 10; k++) { off[k] = pos; pos += al(sizes[k]); }
    off[10] = pos;
    DevBuf<unsigned char>& blob = ctx->tab_blob[(size_t)s];
    CD_CUDA(ctx, blob.ensure(pos));
    // raw columns on the device (scratch of this call)
    DevBuf<int32_t> d_bait, d_oe, d_tblb, d_tlb, d_N, d_cb, d_co;
    DevBuf<double> d_sj, d_si, d_tm;
    DevBuf<unsigned long long> best, k0, k1;
    DevBuf<unsigned int> i0, i1;
    DevBuf<unsigned char> tmp;
    const size_t ms = (size_t)m, mcs = (size_t)mc;
    CD_CUDA(ctx, d_bait.ensure(ms)); CD_CUDA(ctx, d_oe.ensure(ms)); CD_CUDA(ctx, d_tblb.ensure(ms)); CD_CUDA(ctx, d_tlb.ensure(ms));
    CD_CUDA(ctx, d_sj.ensure(ms)); CD_CUDA(ctx, d_si.ensure(ms)); CD_CUDA(ctx, d_tm.ensure(ms));
    CD_CUDA(ctx, best.ensure(2 * (size_t)F + 2 * nt));
    CD_CUDA(ctx, ctx->asm_status.ensure(1));
    CD_CUDA(ctx, cudaMemsetAsync(ctx->asm_status.p, 0, sizeof(int32_t), st));
    if (m > 0) {
        CD_CUDA(ctx, cudaMemcpyAsync(d_bait.p, t->baitID, sizeof(int32_t) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_oe.p, t->otherEndID, sizeof(int32_t) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_tblb.p, t->tblb, sizeof(int32_t) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_tlb.p, t->tlb, sizeof(int32_t) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_sj.p, t->s_j, sizeof(double) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_si.p, t->s_i, sizeof(double) * ms, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_tm.p, t->Tmean, sizeof(double) * ms, cudaMemcpyHostToDevice, st));
    }
    CD_LAUNCHN(ctx, m > 0 ? 2 : 0, tb_launch_first(m, d_bait.p, d_oe.p, d_tblb.p, d_tlb.p, F, ctx->frag_id0, t->n_tblb, t->n_tlb, best.p,
                                                  ctx->asm_status.p, st));
    CD_LAUNCHN(ctx, 1, tb_launch_fill(F, t->n_tblb, t->n_tlb, best.p, d_sj.p, d_tblb.p, d_si.p, d_tlb.p, d_tm.p,
                                      (double*)(blob.p + off[0]), (int32_t*)(blob.p + off[1]), (double*)(blob.p + off[2]),
                                      (int32_t*)(blob.p + off[3]), (double*)(blob.p + off[4]), st));
    CD_CUDA(ctx, cudaMemcpyAsync(blob.p + off[6], t->distfun, sizeof(double) * 10, cudaMemcpyHostToDevice, st));
    // counts: sort the (bait, other end) keys, cut the rows of baits outside the rmap, CSR offsets by lower bound
    const int32_t *cb = d_bait.p, *co = d_oe.p, *cN = nullptr;
    CD_CUDA(ctx, d_N.ensure(mcs));
    if (own_counts) {
        if (m > 0) CD_CUDA(ctx, cudaMemcpyAsync(d_N.p, t->N, sizeof(int32_t) * ms, cudaMemcpyHostToDevice, st));
    } else {
        CD_CUDA(ctx, d_cb.ensure(mcs)); CD_CUDA(ctx, d_co.ensure(mcs));
        CD_CUDA(ctx, cudaMemcpyAsync(d_cb.p, t->cnt_baitID, sizeof(int32_t) * mcs, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_co.p, t->cnt_otherEndID, sizeof(int32_t) * mcs, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(d_N.p, t->cnt_N, sizeof(int32_t) * mcs, cudaMemcpyHostToDevice, st));
        cb = d_cb.p; co = d_co.p;
    }
    cN = d_N.p;
    CD_CUDA(ctx, k0.ensure(mcs)); CD_CUDA(ctx, k1.ensure(mcs)); CD_CUDA(ctx, i0.ensure(mcs)); CD_CUDA(ctx, i1.ensure(mcs));
    int64_t* cnt_off_dev = (int64_t*)(blob.p + off[7]);
    if (mc > 0) {
        CD_LAUNCHN(ctx, 1, tb_launch_count_keys(mc, cb, co, F, ctx->frag_id0, k0.p, i0.p, st));
        size_t bytes = 0;
        CD_CUDA(ctx, cp_sort_pairs_u64(nullptr, bytes, k0.p, k1.p, i0.p, i1.p, mc, st));
        CD_CUDA(ctx, tmp.ensure(bytes));
        CD_LAUNCHN(ctx, 1, cp_sort_pairs_u64(tmp.p, bytes, k0.p, k1.p, i0.p, i1.p, mc, st));
    }
    CD_LAUNCHN(ctx, 1, tb_launch_count_offsets(F, mc, k1.p, cnt_off_dev, st));
    int64_t valid = 0;
    int32_t status = 0;
    CD_CUDA(ctx, cudaMemcpyAsync(&valid, cnt_off_dev + F, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(&status, ctx->asm_status.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    if (status & 1) return ctx->fail(CD_EINVAL, "cd_build_sample_tables: a baitID / otherEndID of the CHiCAGO table is not a fragment of the rmap");
    if (status & 2) return ctx->fail(CD_EINVAL, "cd_build_sample_tables: a tblb / tlb code is outside [0, n_tblb) x [0, n_tlb)");
    CD_LAUNCHN(ctx, valid > 0 ? 1 : 0, tb_launch_count_gather(valid, k1.p, i1.p, cN, (int32_t*)(blob.p + off[8]), (int32_t*)(blob.p + off[9]), st));
    AssembleTables& a = ctx->tabs_host[(size_t)s];
    a.s_j = (const double*)(blob.p + off[0]); a.tblb = (const int32_t*)(blob.p + off[1]);
    a.s_i = (const double*)(blob.p + off[2]); a.tlb = (const int32_t*)(blob.p + off[3]);
    a.tmean = (const double*)(blob.p + off[4]); a.tmin = (const double*)(blob.p + off[5]);
    a.distfun = (const double*)(blob.p + off[6]); a.cnt_off = (const int64_t*)(blob.p + off[7]);
    a.cnt_oe = (const int32_t*)(blob.p + off[8]); a.cnt_N = (const int32_t*)(blob.p + off[9]);
    a.n_tblb = t->n_tblb; a.n_tlb = t->n_tlb;
    CD_LAUNCHN(ctx, 1, launch_tmin(t->n_tblb, t->n_tlb, a.tmean, (double*)(blob.p + off[5]), st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));       // the scratch columns of this call are freed on return
    ctx->tab_set[(size_t)s] = 1;
    ctx->have_agg = false;
    return CD_OK;
}

int cd_get_sample_tables(cd_ctx* ctx, int s, double* s_j, int32_t* tblb, double* s_i, int32_t* tlb, double* tmean,
                         int64_t* cnt_off, int32_t* cnt_oe, int32_t* cnt_N)
{
    if (!ctx) return CD_EINVAL;
    if (s < 0 || s >= (int)ctx->tab_set.size() || !ctx->tab_set[(size_t)s])
        return ctx->fail(CD_EINVAL, "cd_get_sample_tables: tables of replicate %d were never set", s);
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    if (ctx->tab_copy_pending) { CD_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_tab_copy, 0)); ctx->tab_copy_pending = false; }
    const AssembleTables& a = ctx->tabs_host[(size_t)s];
    const size_t F = (size_t)ctx->F, nt = (size_t)a.n_tblb * (size_t)a.n_tlb;
    int64_t ncnt = 0;
    CD_CUDA(ctx, cudaMemcpyAsync(&ncnt, a.cnt_off + F, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    if (s_j) CD_CUDA(ctx, cudaMemcpyAsync(s_j, a.s_j, sizeof(double) * F, cudaMemcpyDeviceToHost, st));
    if (tblb) CD_CUDA(ctx, cudaMemcpyAsync(tblb, a.tblb, sizeof(int32_t) * F, cudaMemcpyDeviceToHost, st));
    if (s_i) CD_CUDA(ctx, cudaMemcpyAsync(s_i, a.s_i, sizeof(double) * F, cudaMemcpyDeviceToHost, st));
    if (tlb) CD_CUDA(ctx, cudaMemcpyAsync(tlb, a.tlb, sizeof(int32_t) * F, cudaMemcpyDeviceToHost, st));
    if (tmean) CD_CUDA(ctx, cudaMemcpyAsync(tmean, a.tmean, sizeof(double) * nt, cudaMemcpyDeviceToHost, st));
    if (cnt_off) CD_CUDA(ctx, cudaMemcpyAsync(cnt_off, a.cnt_off, sizeof(int64_t) * (F + 1), cudaMemcpyDeviceToHost, st));
    if (cnt_oe && ncnt > 0) CD_CUDA(ctx, cudaMemcpyAsync(cnt_oe, a.cnt_oe, sizeof(int32_t) * (size_t)ncnt, cudaMemcpyDeviceToHost, st));
    if (cnt_N && ncnt > 0) CD_CUDA(ctx, cudaMemcpyAsync(cnt_N, a.cnt_N, sizeof(int32_t) * (size_t)ncnt, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    return CD_OK;
}

int cd_assemble(cd_ctx* ctx, int keep_rows, int32_t* K_out, double* fullmean_out, double* avDist_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions || !ctx->have_region_rows || !ctx->have_rmap)
        return ctx->fail(CD_EINVAL, "cd_assemble: needs cd_set_rmap, cd_set_regions and cd_set_region_rows");
    const int S = ctx->des.S;
    if ((int)ctx->tab_set.size() != S) return ctx->fail(CD_EINVAL, "cd_assemble: no replicate tables set");
    for (int s = 0; s < S; s++)
        if (!ctx->tab_set[(size_t)s]) return ctx->fail(CD_EINVAL, "cd_assemble: tables of replicate %d were never set", s);
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t n = ctx->n, R = ctx->R;
    CD_CUDA(ctx, ctx->K.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, ctx->FM.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, ctx->avDist.ensure((size_t)n));
    CD_CUDA(ctx, ctx->asm_status.ensure(1));
    CD_CUDA(ctx, ctx->tabs_dev.ensure(sizeof(AssembleTables) * (size_t)S));
    if (keep_rows) {
        if (ctx->rows_borrowed) return ctx->fail(CD_EINVAL, "cd_assemble: rows were set with cd_set_rows_device");
        CD_CUDA(ctx, ctx->N_rows.ensure((size_t)S * (size_t)R));
        CD_CUDA(ctx, ctx->FM_rows.ensure((size_t)S * (size_t)R));
        CD_CUDA(ctx, ctx->BM_rows.ensure((size_t)S * (size_t)R));
        CD_CUDA(ctx, cudaStreamSynchronize(ctx->st_copy));          // no upload may still target the buffer written here
        std::fill(ctx->staged.begin(), ctx->staged.end(), 0);
        ctx->front = 0; ctx->front_used = true;
        ctx->N_rows_p = ctx->N_rows.p; ctx->FM_rows_p = ctx->FM_rows.p;
    }
    ctx->have_bm_rows = keep_rows != 0;
    if (ctx->tab_copy_pending) { CD_CUDA(ctx, cudaStreamWaitEvent(ctx->st, ctx->ev_tab_copy, 0)); ctx->tab_copy_pending = false; }
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->tabs_dev.p, ctx->tabs_host.data(), sizeof(AssembleTables) * (size_t)S, cudaMemcpyHostToDevice, ctx->st));
    CD_CUDA(ctx, cudaMemsetAsync(ctx->asm_status.p, 0, sizeof(int32_t), ctx->st));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->st));
    CD_LAUNCHN(ctx, n > 0 ? 1 : 0, launch_assemble(n, S, ctx->row_off.p, R, ctx->row_bait.p, ctx->row_oe.p, ctx->F, ctx->frag_id0,
                                                  ctx->frag_chr.p, ctx->frag_start.p, ctx->frag_end.p,
                                                  (const AssembleTables*)ctx->tabs_dev.p, ctx->K.p, ctx->FM.p, ctx->avDist.p,
                                                  keep_rows ? ctx->N_rows.p : nullptr, keep_rows ? ctx->FM_rows.p : nullptr,
                                                  keep_rows ? ctx->BM_rows.p : nullptr, ctx->asm_status.p, ctx->st));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->st));
    int32_t status = 0;
    CD_CUDA(ctx, cudaMemcpyAsync(&status, ctx->asm_status.p, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->st));
    if (K_out) CD_CUDA(ctx, cudaMemcpyAsync(K_out, ctx->K.p, sizeof(int32_t) * (size_t)S * (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    if (fullmean_out) CD_CUDA(ctx, cudaMemcpyAsync(fullmean_out, ctx->FM.p, sizeof(double) * (size_t)S * (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    if (avDist_out) CD_CUDA(ctx, cudaMemcpyAsync(avDist_out, ctx->avDist.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    if (status & 1) return ctx->fail(CD_EINVAL, "cd_assemble: a region row names a fragment outside the rmap");
    if (status & 2) return ctx->fail(CD_EINVAL, "cd_assemble: a region's rows do not share one baitID");
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->timings[0] = ms;
    if (keep_rows) std::fill(ctx->sample_set.begin(), ctx->sample_set.end(), 1);
    ctx->have_agg = true;
    return CD_OK;
}

int cd_get_sample_rows(cd_ctx* ctx, int s, int32_t* N_out, double* fullmean_out)
{
    if (!ctx) return CD_EINVAL;
    const int S = ctx->des.S;
    if (s < 0 || s >= S || !ctx->have_regions || (!ctx->N_rows_p && !ctx->staged[(size_t)s]) || ctx->rows_borrowed || !ctx->sample_set[(size_t)s])
        return ctx->fail(CD_EINVAL, "cd_get_sample_rows: no per-row columns on the device (cd_assemble with keep_rows, or cd_set_sample_rows)");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t R = (size_t)ctx->R;
    const int32_t* Np = ctx->N_rows_p;
    const double* Fp = ctx->FM_rows_p;
    if (ctx->staged[(size_t)s]) {               // uploaded since the last aggregation: still in the staging buffer
        CD_CUDA(ctx, cudaStreamSynchronize(ctx->st_copy));
        Np = ctx->nbuf(ctx->back()); Fp = ctx->fbuf(ctx->back());
    }
    if (N_out) CD_CUDA(ctx, cudaMemcpyAsync(N_out, Np + (size_t)s * R, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, ctx->st));
    if (fullmean_out) CD_CUDA(ctx, cudaMemcpyAsync(fullmean_out, Fp + (size_t)s * R, sizeof(double) * R, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    return CD_OK;
}

int cd_get_sample_bmean(cd_ctx* ctx, int s, double* bmean_out)
{
    if (!ctx) return CD_EINVAL;
    if (s < 0 || s >= ctx->des.S || !ctx->have_bm_rows || !bmean_out)
        return ctx->fail(CD_EINVAL, "cd_get_sample_bmean: needs cd_assemble with keep_rows");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t R = (size_t)ctx->R;
    CD_CUDA(ctx, cudaMemcpyAsync(bmean_out, ctx->BM_rows.p + (size_t)s * R, sizeof(double) * R, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    return CD_OK;
}

int cd_aggregate(cd_ctx* ctx, int32_t* K_out, double* fullmean_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_regions) return ctx->fail(CD_EINVAL, "cd_aggregate: call cd_set_regions first");
    const int S = ctx->des.S;
    for (int s = 0; s < S; s++)
        if (!ctx->sample_set[(size_t)s]) return ctx->fail(CD_EINVAL, "cd_aggregate: rows of sample %d were never set", s);
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t n = ctx->n;
    CD_CUDA(ctx, ctx->K.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, ctx->FM.ensure((size_t)S * (size_t)n));
    if (!ctx->rows_borrowed) {
        int n_staged = 0;
        for (uint8_t f : ctx->staged) n_staged += f ? 1 : 0;
        if (n_staged > 0) {
            const int b = ctx->back();
            CD_CUDA(ctx, cudaStreamWaitEvent(ctx->st, ctx->ev_copy, 0));
            if (b != ctx->front || !ctx->front_used) {
                // samples that were not uploaded again keep the rows of the previous batch
                if (ctx->front_used && n_staged < S) {
                    const size_t R = (size_t)ctx->R;
                    for (int s = 0; s < S; s++) if (!ctx->staged[(size_t)s]) {
                        CD_CUDA(ctx, cudaMemcpyAsync(ctx->nbuf(b) + (size_t)s * R, ctx->nbuf(ctx->front) + (size_t)s * R, sizeof(int32_t) * R, cudaMemcpyDeviceToDevice, ctx->st));
                        CD_CUDA(ctx, cudaMemcpyAsync(ctx->fbuf(b) + (size_t)s * R, ctx->fbuf(ctx->front) + (size_t)s * R, sizeof(double) * R, cudaMemcpyDeviceToDevice, ctx->st));
                    }
                }
                ctx->front = b;
            }
            ctx->front_used = true;
            std::fill(ctx->staged.begin(), ctx->staged.end(), 0);
        }
        ctx->N_rows_p = ctx->nbuf(ctx->front); ctx->FM_rows_p = ctx->fbuf(ctx->front);
    }
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[0], ctx->st));
    CD_LAUNCHN(ctx, n > 0 ? 1 : 0, launch_aggregate(n, S, ctx->row_off.p, ctx->R, ctx->N_rows_p, ctx->FM_rows_p, ctx->K.p, ctx->FM.p, ctx->st));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[1], ctx->st));
    if (!ctx->rows_borrowed) CD_CUDA(ctx, cudaEventRecord(ctx->ev_read[ctx->front], ctx->st));
    if (K_out) CD_CUDA(ctx, cudaMemcpyAsync(K_out, ctx->K.p, sizeof(int32_t) * (size_t)S * (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    if (fullmean_out) CD_CUDA(ctx, cudaMemcpyAsync(fullmean_out, ctx->FM.p, sizeof(double) * (size_t)S * (size_t)n, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->timings[0] = ms;
    ctx->have_agg = true;
    return CD_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// global steps
// ---------------------------------------------------------------------------------------------
namespace {

// R median() of the finite entries of B columns (column c at base + c*stride, n local values each, optionally
// transformed to |x - center[c]|) over ALL ranks -> out_dev[c] = scale * median (exp'ed if do_exp): one cooperative
// kernel; in a sharded run it all-reduces its 2048-bin counters through peer memory itself.
int medians(cd_ctx* ctx, const double* base, int64_t stride, int64_t n, int B, const double* center_dev,
            double* out_dev, int do_exp, double scale)
{
    CD_CUDA(ctx, ctx->sel_state.ensure((size_t)kSelP2PMaxCols * kSelStateHost));
    CD_CUDA(ctx, ctx->sel_hist.ensure((size_t)kSelP2PMaxCols * kSelBinsHost));
    CD_CUDA(ctx, ctx->sel_aux.ensure((size_t)kSelP2PMaxCols * 3));
    SelP2P pp{};
    pp.nranks = 1;
    pp.err = ctx->counters.p + kCntErr;
    if (ctx->comm.active()) {
        pp.nranks = ctx->comm.nranks; pp.rank = ctx->comm.rank;
        pp.peers = ctx->sel_peers_dev.p; pp.mymail = ctx->sel_mail.p;
        pp.seq = ctx->sel_seq + 1;
        ctx->sel_seq += kSelExchanges;
    }
    CD_LAUNCHN(ctx, 1, sel_launch_fused(n, B, base, stride, center_dev, out_dev, do_exp, scale, ctx->sel_state.p, ctx->sel_hist.p,
                                        ctx->sel_aux.p, reinterpret_cast<unsigned int*>(ctx->counters.p + kCntSelBar), pp, ctx->st));
    return CD_OK;
}

// after a host sync that follows a global step: did a peer-memory exchange give up?
int check_peer_exchange(cd_ctx* ctx, unsigned long long err_word)
{
    if (err_word == 0ull) return CD_OK;
    cudaMemsetAsync(ctx->counters.p + kCntErr, 0, sizeof(unsigned long long), ctx->st);
    return ctx->fail(CD_ECOMM, "peer-memory exchange timed out: another rank stopped before reaching the same step");
}

// estimateSizeFactors over ALL regions of all ranks -> scal[0..S)
int size_factors(cd_ctx* ctx, double* sf_host)
{
    const int S = ctx->des.S;
    const int64_t n = ctx->n;
    // zeroed at the start of every cd_region_test
    double* bad_dev = reinterpret_cast<double*>(ctx->counters.p + kCntBad);
    CD_CUDA(ctx, ctx->g_LR.ensure((size_t)S * (size_t)n));
    CD_LAUNCHN(ctx, 1, launch_log_ratios(n, S, ctx->K.p, ctx->g_LR.p, bad_dev, ctx->st));
    int rc = medians(ctx, ctx->g_LR.p, n, n, S, nullptr, ctx->scal.p + kScalSf, 1, 1.0);
    if (rc != CD_OK) return rc;
    // every rank must refuse together, or the clean ones would wait for the others in the next collective
    CD_COMM(ctx, ctx->comm.allreduce_sum(bad_dev, 1, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinSf, ctx->scal.p + kScalSf, sizeof(double) * S, cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinErr, ctx->counters.p + kCntErr, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinBad, bad_dev, sizeof(double), cudaMemcpyDeviceToHost, ctx->st));
    CD_CUDA(ctx, cudaStreamSynchronize(ctx->st));
    unsigned long long errw;
    memcpy(&errw, ctx->h_pinned + kPinErr, sizeof(errw));
    if ((rc = check_peer_exchange(ctx, errw)) != CD_OK) return rc;
    if (ctx->h_pinned[kPinBad] != 0.0)
        return ctx->fail(CD_EINVAL, "NA or negative values in the count matrix (DESeq2: \"NA values are not allowed in the count "
                                    "matrix\" / \"some values in assay are negative\"); NA_integer_ marks a region sum beyond "
                                    "the int32 range");
    for (int s = 0; s < S; s++) {
        sf_host[s] = ctx->h_pinned[kPinSf + s];
        if (std::isnan(sf_host[s]))
            return ctx->fail(CD_ENUMERIC, "every gene contains at least one zero, cannot compute log geometric means");
    }
    return CD_OK;
}

// Timing section 2: one line search of a batch (gene-wise without a prior, MAP with one), then the count of its
// posterior evaluations, which cd_last_search_counts reports per call.
int timed_fit_disp(cd_ctx* ctx, int64_t nv, int64_t n, int S, int p, const CdDesign* des_dev, const int32_t* K,
                   const double* prior_log_mean, const BatchScalars& prior_sigmasq, int32_t* iter)
{
    cudaStream_t st = ctx->st;
    ctx->tm_begin(2);
    CD_LAUNCHN(ctx, 2, launch_fit_disp(nv, n, S, p, des_dev, K, ctx->mu.p, ctx->start_log.p, prior_log_mean, prior_sigmasq,
                                       ctx->log_alpha.p, iter, ctx->initial_lp.p, ctx->last_lp.p,
                                       ctx->counters.p + kCntFitDispQueue, ctx->park, st));
    ctx->tm_end();
    if (ctx->n_eval_calls < 16 && nv > 0) {
        count_evals_kernel<<<592, 256, 0, st>>>(nv, iter, ctx->eval_counts.p + ctx->n_eval_calls);
        ctx->launches++;
        ctx->eval_call_p[ctx->n_eval_calls] = p; ctx->eval_call_regions[ctx->n_eval_calls] = nv; ctx->n_eval_calls++;
    }
    return CD_OK;
}

// Timing section 4: the grid refit of the rows the preceding gene_post / map_post listed.
int timed_grid_refit(cd_ctx* ctx, int64_t nv, int64_t n, int S, int p, const CdDesign* des_dev, const int32_t* K,
                     const double* prior_mean_disp, const BatchScalars& prior_sigmasq, int grid_len, double* disp_out,
                     double* dispersion_out, const uint8_t* flags, const double* dispGeneEst)
{
    ctx->tm_begin(4);
    CD_LAUNCHN(ctx, 1, launch_fit_disp_grid(nv, n, S, p, des_dev, ctx->refit_count.p, ctx->refit_list.p, K, ctx->mu.p,
                                            prior_mean_disp, prior_sigmasq, grid_len, disp_out, dispersion_out, flags,
                                            dispGeneEst, ctx->st));
    ctx->tm_end();
    return CD_OK;
}

struct BatchOut { double a0[kMaxBatch], a1[kMaxBatch], varLogDispEsts[kMaxBatch], dispPriorVar[kMaxBatch], sum_deviance[kMaxBatch]; };

// estimateDispersions + nbinomWaldTest for a batch of G fits of one design that differ in their normalisation
// (mode, theta[g]): the theta grid (G = 5, design ~ 1, only the total deviances are wanted) or the final fit (G = 1).
// All per-region arrays of the batch are indexed by the virtual region g * n + i.
int run_batch(cd_ctx* ctx, const CdDesign& des, const CdDesign* des_dev, int G, int mode, const double* theta,
              double prior_var_override, int grid_len, bool final_fit, BatchOut& bo, const cd_options* opt)
{
    const int S = des.S, p = des.p;
    const int64_t n = ctx->n, nv = (int64_t)G * n;
    cudaStream_t st = ctx->st;
    const int df = S - p;
    // S - p <= 3: DESeq2's seeded Monte-Carlo rule -- the caller's function if one is given (an R front end evaluates
    // DESeq2's own code there), else the library's restatement of it (priorvar.cpp)
    const bool ask_caller = std::isnan(prior_var_override) && df <= 3 && opt && opt->prior_var_fn;
    const bool small_df_rule = std::isnan(prior_var_override) && df <= 3 && !ask_caller;
    const int32_t* K = (G > 1) ? ctx->Kb.p : ctx->K.p;
    double* baseMean = ctx->g_baseMean.p;
    double* dispGeneEst = ctx->g_dispGeneEst.p;
    double* dispFit = ctx->g_dispFit.p;
    uint8_t* flags = ctx->g_flags.p;
    double* sf_dev = ctx->scal.p + kScalSf;
    double* sums_dev = ctx->scal.p + kScalSums;
    double* xim_dev = ctx->scal.p + kScalXim;
    double* trend_dev = ctx->scal.p + kScalTrend;
    unsigned long long* err_dev = ctx->counters.p + kCntErr;

    BatchScalars th{};
    for (int g = 0; g < G; g++) th.v[g] = theta[g];
    CD_LAUNCHN(ctx, 1, launch_norm_factors(n, S, G, ctx->FM.p, sf_dev, mode, th, ctx->nf.p, ctx->K.p, G > 1 ? ctx->Kb.p : nullptr, st));
    CD_LAUNCHN(ctx, 1, launch_base_stats(nv, S, des_dev, K, ctx->nf.p, baseMean, ctx->baseVar.p, ctx->rough.p, flags,
                                         des.linear_mu ? ctx->mu.p : nullptr, st));
    CD_LAUNCHN(ctx, 2, launch_masked_colsums(n, G, S, ctx->nf.p, flags, ctx->partial.p, sums_dev, st));
    CD_COMM(ctx, ctx->comm.allreduce_sum(sums_dev, (size_t)G * (S + 1), st));
    CD_LAUNCHN(ctx, 1, launch_xim(G, S, sums_dev, xim_dev, st));
    CD_LAUNCHN(ctx, 1, launch_gene_init(nv, n, S, baseMean, ctx->baseVar.p, ctx->rough.p, flags, xim_dev, ctx->alpha_init.p,
                                        ctx->start_log.p, st));
    if (!des.linear_mu) {
        // mu from an NB GLM fitted with the rough dispersion (fitNbinomGLMs(alpha_hat = alpha_init)$mu)
        CD_LAUNCHN(ctx, 3, launch_wald(nv, S, p, des_dev, K, ctx->nf.p, ctx->alpha_init.p, flags, ctx->wald_ws, nullptr, nullptr,
                                       nullptr, nullptr, nullptr, nullptr, nullptr, ctx->mu.p, st));
    }
    BatchScalars none{};
    for (int g = 0; g < kMaxBatch; g++) none.v[g] = 1.0;
    int rc = timed_fit_disp(ctx, nv, n, S, p, des_dev, K, nullptr, none, ctx->dispGeneIter.p);
    if (rc != CD_OK) return rc;
    CD_LAUNCHN(ctx, 1, launch_gene_post(nv, S, ctx->alpha_init.p, ctx->log_alpha.p, ctx->dispGeneIter.p, ctx->initial_lp.p,
                                        ctx->last_lp.p, flags, dispGeneEst, ctx->refit_list.p, ctx->refit_count.p, st));
    rc = timed_grid_refit(ctx, nv, n, S, p, des_dev, K, nullptr, none, grid_len, dispGeneEst, nullptr, flags, dispGeneEst);
    if (rc != CD_OK) return rc;
    // trend + MAD of every fit over the regions of all ranks.  Nothing is gathered: the trend passes all-reduce 8 sums
    // per fit, the medians all-reduce histogram counters, both inside their kernels.  One host sync for both.
    ctx->tm_begin(5);
    const bool trend_given = final_fit && opt && opt->trend_a0 > 0.0 && opt->trend_a1 > 0.0;
    const bool vld_given = final_fit && opt && opt->var_log_disp > 0.0;
    if (trend_given) {
        double* h = ctx->h_pinned + kPinTrendIn;
        for (int g = 0; g < G; g++) { h[8 * g] = opt->trend_a0; h[8 * g + 1] = opt->trend_a1; h[8 * g + 2] = 0.0; h[8 * g + 3] = 0.0; h[8 * g + 4] = 0.0; }
        CD_CUDA(ctx, cudaMemcpyAsync(trend_dev, h, sizeof(double) * 8 * G, cudaMemcpyHostToDevice, st));
    } else {
        // one cooperative kernel; in a sharded run it all-reduces the sums of every pass through peer memory
        TrendP2P pp{};
        pp.nranks = ctx->comm.active() ? ctx->comm.nranks : 1;
        pp.rank = ctx->comm.rank;
        pp.peers = ctx->p2p_peers_dev.p; pp.mymail = ctx->p2p_mail.p;
        pp.epoch = ++ctx->p2p_epoch;
        pp.err = err_dev;
        pp.wait_cycles = ctx->comm.active() ? ctx->counters.p + kCntWait : nullptr;
        CD_LAUNCHN(ctx, 1, launch_trend_fit(n, G, baseMean, dispGeneEst, flags, ctx->trend_xs.p, ctx->partial.p,
                                            reinterpret_cast<unsigned int*>(ctx->counters.p + kCntTrendBar), trend_dev, pp, st));
    }
    CD_LAUNCHN(ctx, 1, launch_trend_apply(nv, n, baseMean, dispGeneEst, flags, trend_dev, dispFit, ctx->g_resid.p,
                                          ctx->start_log.p, ctx->log_fit.p, st));
    rc = medians(ctx, ctx->g_resid.p, n, n, G, nullptr, ctx->scal.p + kScalMed, 0, 1.0);
    if (rc != CD_OK) return rc;
    rc = medians(ctx, ctx->g_resid.p, n, n, G, ctx->scal.p + kScalMed, ctx->scal.p + kScalMad, 0, 1.4826);
    if (rc != CD_OK) return rc;
    ctx->tm_end();
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinTrend, trend_dev, sizeof(double) * 8 * G, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinMad, ctx->scal.p + kScalMad, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinErr, err_dev, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    unsigned long long errw;
    memcpy(&errw, ctx->h_pinned + kPinErr, sizeof(errw));
    if ((rc = check_peer_exchange(ctx, errw)) != CD_OK) return rc;
    BatchScalars prior{}, thr{};
    for (int g = 0; g < kMaxBatch; g++) { prior.v[g] = 1.0; thr.v[g] = 0.0; }
    for (int g = 0; g < G; g++) {
        const double* t = ctx->h_pinned + kPinTrend + 8 * g;
        const int tstatus = (int)t[2];
        if (tstatus == 6) return check_peer_exchange(ctx, 1ull);
        if (tstatus != 0) {
            static const char* why[] = {"", "fewer than 2 usable regions", "invalid starting values", "no valid step",
                                        "non-positive coefficients", "did not converge"};
            return ctx->fail(CD_ENUMERIC, "parametric dispersion fit failed (%s); the reference would switch to a local "
                                          "regression fit (locfit), which is not implemented", why[tstatus < 6 ? tstatus : 0]);
        }
        const double mad = ctx->h_pinned[kPinMad + g];
        if (std::isnan(mad) && !vld_given)
            return ctx->fail(CD_ENUMERIC, "all gene-wise dispersion estimates are within 2 orders of magnitude of the minimum");
        const double varLogDispEsts = vld_given ? opt->var_log_disp : mad * mad;
        double dispPriorVar;
        if (!std::isnan(prior_var_override)) dispPriorVar = prior_var_override;
        else if (ask_caller) {
            // the residuals are in g_resid (+inf where the region is excluded); the caller's rule sees the finite ones
            if (ctx->comm.active() && ctx->comm.nranks > 1)
                return ctx->fail(CD_EINVAL, "prior_var_fn needs the residuals of all regions: not available in a sharded run, pass "
                                            "disp_prior_var");
            std::vector<double> resid((size_t)n);
            CD_CUDA(ctx, cudaMemcpyAsync(resid.data(), ctx->g_resid.p + (size_t)g * n, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
            CD_CUDA(ctx, cudaStreamSynchronize(st));
            size_t m = 0;
            for (size_t i = 0; i < (size_t)n; i++) if (std::isfinite(resid[i])) resid[m++] = resid[i];
            dispPriorVar = opt->prior_var_fn(opt->prior_var_user, df, (int64_t)m, resid.data());
            if (!(dispPriorVar > 0.0) || !std::isfinite(dispPriorVar))
                return ctx->fail(CD_ENUMERIC, "prior_var_fn returned %g for df = %d (%lld residuals)", dispPriorVar, df, (long long)m);
        } else if (small_df_rule) {
            // the rule needs the histogram of the residuals only, and bin counts add up over shards
            std::vector<double> resid((size_t)n);
            CD_CUDA(ctx, cudaMemcpyAsync(resid.data(), ctx->g_resid.p + (size_t)g * n, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
            CD_CUDA(ctx, cudaStreamSynchronize(st));
            size_t m = 0;
            for (size_t i = 0; i < (size_t)n; i++) if (std::isfinite(resid[i])) resid[m++] = resid[i];
            double counts[40];
            cd_prior_var_hist((int64_t)m, resid.data(), counts);
            if (ctx->comm.active() && ctx->comm.nranks > 1) {
                double* c_dev = ctx->scal.p + kScalSums;                  // (free again at this point of the fit)
                CD_CUDA(ctx, cudaMemcpyAsync(c_dev, counts, sizeof(counts), cudaMemcpyHostToDevice, st));
                CD_COMM(ctx, ctx->comm.allreduce_sum(c_dev, 40, st));
                CD_CUDA(ctx, cudaMemcpyAsync(counts, c_dev, sizeof(counts), cudaMemcpyDeviceToHost, st));
                CD_CUDA(ctx, cudaStreamSynchronize(st));
            }
            dispPriorVar = cd_prior_var_from_hist(df, counts);
            if (!(dispPriorVar > 0.0) || !std::isfinite(dispPriorVar))
                return ctx->fail(CD_ENUMERIC, "dispersion prior variance for S - p = %d: no residual inside (-10, 10) to match", df);
        } else dispPriorVar = std::max(varLogDispEsts - trigamma_host(df / 2.0), 0.25);
        bo.a0[g] = t[0]; bo.a1[g] = t[1]; bo.varLogDispEsts[g] = varLogDispEsts; bo.dispPriorVar[g] = dispPriorVar;
        if (g == 0 || t[4] > ctx->trend_passes_batch) ctx->trend_passes_batch = t[4];
        prior.v[g] = dispPriorVar;
        thr.v[g] = 2.0 * sqrt(varLogDispEsts);
    }

    ctx->trend_passes += ctx->trend_passes_batch;          // the fits of a batch advance in lock step: max over the fits
    ctx->trend_passes_batch = 0;

    // MAP
    rc = timed_fit_disp(ctx, nv, n, S, p, des_dev, K, ctx->log_fit.p, prior, ctx->dispIter.p);
    if (rc != CD_OK) return rc;
    CD_LAUNCHN(ctx, 1, launch_map_post(nv, n, S, ctx->log_alpha.p, ctx->dispIter.p, dispGeneEst, dispFit, thr,
                                       flags, ctx->dispMAP.p, ctx->dispersion.p, ctx->refit_list.p, ctx->refit_count.p, st));
    rc = timed_grid_refit(ctx, nv, n, S, p, des_dev, K, dispFit, prior, grid_len, ctx->dispMAP.p, ctx->dispersion.p, flags,
                          dispGeneEst);
    if (rc != CD_OK) return rc;
    // NB GLM + Wald (final fit) / total deviance only (theta-grid fits)
    ctx->tm_begin(3);
    if (final_fit) {
        CD_LAUNCHN(ctx, p > 1 ? 3 : 2, launch_wald(nv, S, p, des_dev, K, ctx->nf.p, ctx->dispersion.p, flags, ctx->wald_ws, ctx->beta.p,
                                                   ctx->betaSE.p, ctx->stat.p, ctx->pvalue.p, ctx->deviance.p, ctx->maxCooks.p,
                                                   ctx->betaIter.p, nullptr, st));
    } else {
        CD_LAUNCHN(ctx, 1, launch_wald_deviance_p1(nv, S, K, ctx->nf.p, ctx->dispersion.p, flags, ctx->lfact.p, ctx->deviance.p, st));
    }
    ctx->tm_end();
    CD_LAUNCHN(ctx, 2, launch_segment_sums(n, G, ctx->deviance.p, ctx->partial.p, ctx->scal.p + kScalDev, st));
    CD_COMM(ctx, ctx->comm.allreduce_sum(ctx->scal.p + kScalDev, (size_t)G, st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + kPinDev, ctx->scal.p + kScalDev, sizeof(double) * G, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    for (int g = 0; g < G; g++) bo.sum_deviance[g] = ctx->h_pinned[kPinDev + g];
    return CD_OK;
}

template <typename T>
int d2h(cd_ctx* ctx, T* dst, const T* src, size_t count)
{
    if (!dst || count == 0) return CD_OK;
    CD_CUDA(ctx, cudaMemcpyAsync(dst, src, sizeof(T) * count, cudaMemcpyDeviceToHost, ctx->st));
    return CD_OK;
}

}  // namespace

extern "C" {

int cd_region_test(cd_ctx* ctx, const cd_options* opt, cd_results* out)
{
    if (!ctx) return CD_EINVAL;
    if (!opt || !out) return ctx->fail(CD_EINVAL, "cd_region_test: null options / results");
    if (!ctx->have_agg) return ctx->fail(CD_EINVAL, "cd_region_test: call cd_aggregate (or cd_set_aggregated) first");
    ctx->have_results = false;
    if (opt->norm < 0 || opt->norm > 2) return ctx->fail(CD_EINVAL, "DESeq2Wrap error: Unknown normalisation method.");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    const int S = ctx->des.S, p = ctx->des.p;
    const int64_t n = ctx->n;
    cudaStream_t st = ctx->st;
    const int grid_len = opt->disp_grid_len > 0 ? opt->disp_grid_len : 20;
    if (grid_len < 2 || grid_len > 32) return ctx->fail(CD_EINVAL, "disp_grid_len must be in [2, 32]");

    // shard geometry
    CD_COMM(ctx, ctx->comm.allgather_i64(n, ctx->shard_n, st));
    ctx->shard_off.assign(ctx->shard_n.size(), 0);
    int64_t tot = 0;
    for (size_t r = 0; r < ctx->shard_n.size(); r++) { ctx->shard_off[r] = tot; tot += ctx->shard_n[r]; }
    ctx->n_tot = tot;                  // regions over all ranks (for reporting; nothing is gathered)
    ctx->g_off = 0;
    if (tot > 2147483647LL) return ctx->fail(CD_EINVAL, "more than 2^31-1 regions in total");
    if (tot < 1) return ctx->fail(CD_EINVAL, "cd_region_test: no regions");

    int norm = opt->norm;
    double theta = opt->theta;
    if (!std::isnan(theta)) {
        // chicdiff.R:1511-1521: theta = 1 is "standard", theta = 0 is "fullmean"
        if (theta == 1.0 && norm != CD_NORM_STANDARD) norm = CD_NORM_STANDARD;
        if (theta == 0.0 && norm != CD_NORM_FULLMEAN) norm = CD_NORM_FULLMEAN;
    }
    static const double default_grid[5] = {0.0, 0.25, 0.5, 0.75, 1.0};
    const bool use_grid = (norm == CD_NORM_COMBINED && std::isnan(theta));
    const double* grid = opt->theta_grid ? opt->theta_grid : default_grid;
    const int ng = opt->theta_grid ? opt->n_theta_grid : 5;
    if (use_grid && (ng < 1 || ng > kMaxBatch)) return ctx->fail(CD_EINVAL, "theta grid must have 1..%d values", kMaxBatch);
    // the fits of the theta grid run as one batch of ng * n virtual regions
    const int Gmax = use_grid ? ng : 1;
    const int64_t nv = (int64_t)Gmax * n;
    if (nv > 2147483647LL) return ctx->fail(CD_EINVAL, "theta grid size x regions exceeds 2^31-1: shard the regions over more GPUs");

    const size_t sn = (size_t)S * (size_t)nv, vn = (size_t)nv;
    CD_CUDA(ctx, ctx->nf.ensure(sn));
    CD_CUDA(ctx, ctx->mu.ensure(sn));
    if (Gmax > 1) CD_CUDA(ctx, ctx->Kb.ensure(sn));
    CD_CUDA(ctx, ctx->baseVar.ensure(vn)); CD_CUDA(ctx, ctx->rough.ensure(vn));
    CD_CUDA(ctx, ctx->alpha_init.ensure(vn)); CD_CUDA(ctx, ctx->log_alpha.ensure(vn));
    CD_CUDA(ctx, ctx->initial_lp.ensure(vn)); CD_CUDA(ctx, ctx->last_lp.ensure(vn));
    CD_CUDA(ctx, ctx->dispMAP.ensure(vn)); CD_CUDA(ctx, ctx->dispersion.ensure(vn));
    CD_CUDA(ctx, ctx->beta.ensure((size_t)CD_MAXP * (size_t)n)); CD_CUDA(ctx, ctx->betaSE.ensure((size_t)CD_MAXP * (size_t)n));
    CD_CUDA(ctx, ctx->stat.ensure((size_t)n)); CD_CUDA(ctx, ctx->pvalue.ensure((size_t)n));
    CD_CUDA(ctx, ctx->deviance.ensure(vn)); CD_CUDA(ctx, ctx->maxCooks.ensure((size_t)n));
    CD_CUDA(ctx, ctx->dispGeneIter.ensure(vn)); CD_CUDA(ctx, ctx->dispIter.ensure(vn));
    CD_CUDA(ctx, ctx->betaIter.ensure((size_t)n)); CD_CUDA(ctx, ctx->refit_list.ensure(vn));
    CD_CUDA(ctx, ctx->g_baseMean.ensure(vn)); CD_CUDA(ctx, ctx->g_dispGeneEst.ensure(vn));
    CD_CUDA(ctx, ctx->g_dispFit.ensure(vn)); CD_CUDA(ctx, ctx->g_resid.ensure(vn));
    CD_CUDA(ctx, ctx->g_flags.ensure(vn)); CD_CUDA(ctx, ctx->trend_xs.ensure(vn));
    CD_CUDA(ctx, ctx->start_log.ensure(vn)); CD_CUDA(ctx, ctx->log_fit.ensure(vn));
    CD_CUDA(ctx, ctx->partial.ensure((size_t)kReduceBlocks * kMaxBatch * (CD_MAXS + 1)));
    CD_CUDA(ctx, ctx->scal.ensure(kScalSize));
    if (!ctx->counters.p) {
        CD_CUDA(ctx, ctx->counters.ensure(kCntSize));
        CD_CUDA(ctx, cudaMemsetAsync(ctx->counters.p, 0, kCntSize * sizeof(unsigned long long), st));
    }
    CD_CUDA(ctx, ctx->refit_count.ensure(1));
    CD_CUDA(ctx, ctx->wald_c.ensure((size_t)S * (size_t)n));
    CD_CUDA(ctx, ctx->wald_b0.ensure((size_t)CD_MAXP * (size_t)n));
    CD_CUDA(ctx, ctx->wald_b.ensure((size_t)CD_MAXP * (size_t)n));
    CD_CUDA(ctx, ctx->wald_iter.ensure((size_t)n));
    if (!ctx->lfact.p) {
        CD_CUDA(ctx, ctx->lfact.ensure(kLfactN));
        CD_LAUNCHN(ctx, 1, launch_lfact_table(ctx->lfact.p, st));
    }
    ctx->wald_ws.lfact = ctx->lfact.p;
    ctx->wald_ws.cmat = ctx->wald_c.p; ctx->wald_ws.beta0 = ctx->wald_b0.p; ctx->wald_ws.beta_nat = ctx->wald_b.p;
    ctx->wald_ws.iter = ctx->wald_iter.p; ctx->wald_ws.work_counter = ctx->counters.p + kCntWaldQueue;
    {
        const int64_t cap = nv / 4 + 4096;
        CD_CUDA(ctx, ctx->park_row.ensure((size_t)cap));
        CD_CUDA(ctx, ctx->park_d.ensure((size_t)cap * 5));
        CD_CUDA(ctx, ctx->park_i.ensure((size_t)cap * 2));
        FitDispPark& pk = ctx->park;
        pk.capacity = cap; pk.row = ctx->park_row.p;
        pk.a = ctx->park_d.p; pk.lp = pk.a + cap; pk.dlp = pk.lp + cap; pk.kappa = pk.dlp + cap; pk.lp0 = pk.kappa + cap;
        pk.iter = ctx->park_i.p; pk.iter_accept = pk.iter + cap;
        pk.count = ctx->counters.p + kCntPark;
    }

    CD_CUDA(ctx, ctx->eval_counts.ensure(16));
    CD_CUDA(ctx, cudaMemsetAsync(ctx->eval_counts.p, 0, 16 * sizeof(unsigned long long), st));
    CD_CUDA(ctx, cudaMemsetAsync(ctx->counters.p + kCntWait, 0, 4 * sizeof(unsigned long long), st));     // waits, bad counts
    ctx->n_eval_calls = 0;
    ctx->trend_passes = 0;
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[2], st));
    memset(out->sizeFactors, 0, sizeof(out->sizeFactors));
    for (int k = 2; k < 8; k++) ctx->timings[k] = 0.0;
    ctx->ev_used = 0;
    ctx->tm_begin(6);
    int rc = size_factors(ctx, out->sizeFactors);
    if (rc != CD_OK) return rc;
    ctx->tm_end();

    out->n_deviances = 0;
    BatchOut bo{};
    if (use_grid) {
        // chicdiff.R:1633-1647: the ng intercept-only fits, as one batch; only their total deviances are wanted
        rc = run_batch(ctx, ctx->des1, ctx->des_dev.p + 1, ng, CD_NORM_COMBINED, grid, opt->disp_prior_var_grid, grid_len, false, bo, opt);
        if (rc != CD_OK) return rc;
        for (int k = 0; k < ng; k++) {
            out->deviances[k] = bo.sum_deviance[k];
            if (std::isnan(bo.sum_deviance[k]))
                return ctx->fail(CD_ENUMERIC, "theta grid: total deviance is NA (an all-zero region is present and chicdiff.R:1647 "
                                              "sums without na.rm); pass theta explicitly, as chicdiffPipeline does for the control set");
        }
        out->n_deviances = ng;
        int best = -1, nbest = 0;
        for (int k = 0; k < ng; k++) {
            if (best < 0 || out->deviances[k] < out->deviances[best]) { best = k; nbest = 1; }
            else if (out->deviances[k] == out->deviances[best]) nbest++;
        }
        if (nbest != 1) return ctx->fail(CD_ENUMERIC, "theta grid: the minimum total deviance is tied");
        theta = grid[best];
    }
    const double theta_final = std::isnan(theta) ? 0.0 : theta;
    rc = run_batch(ctx, ctx->des, ctx->des_dev.p, 1, norm, &theta_final, opt->disp_prior_var, grid_len, true, bo, opt);
    if (rc != CD_OK) return rc;
    CD_CUDA(ctx, cudaEventRecord(ctx->ev[3], st));
    struct { double a0, a1, varLogDispEsts, dispPriorVar; } po = {bo.a0[0], bo.a1[0], bo.varLogDispEsts[0], bo.dispPriorVar[0]};

    out->theta = (norm == CD_NORM_COMBINED) ? theta : NAN;
    out->trend_a0 = po.a0; out->trend_a1 = po.a1;
    out->varLogDispEsts = po.varLogDispEsts; out->dispPriorVar = po.dispPriorVar;

    CD_CUDA(ctx, cudaMemsetAsync(ctx->counters.p + kCntFlags, 0, 4 * sizeof(unsigned long long), st));
    const uint8_t* flags = ctx->g_flags.p + ctx->g_off;
    if (n > 0) {
        count_flags_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, flags, ctx->counters.p + kCntFlags);
        ctx->launches++;
    }
    unsigned long long hc[4] = {0, 0, 0, 0};
    CD_CUDA(ctx, cudaMemcpyAsync(hc, ctx->counters.p + kCntFlags, sizeof(hc), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->eval_counts_host, ctx->eval_counts.p, sizeof(ctx->eval_counts_host), cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaMemcpyAsync(ctx->wait_host, ctx->counters.p + kCntWait, sizeof(ctx->wait_host), cudaMemcpyDeviceToHost, st));
    const size_t nn = (size_t)n;
    if ((rc = d2h(ctx, out->baseMean, ctx->g_baseMean.p + ctx->g_off, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->baseVar, ctx->baseVar.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispGeneEst, ctx->g_dispGeneEst.p + ctx->g_off, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispFit, ctx->g_dispFit.p + ctx->g_off, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispMAP, ctx->dispMAP.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispersion, ctx->dispersion.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->log2FoldChange, ctx->beta.p + (size_t)(p - 1) * nn, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->lfcSE, ctx->betaSE.p + (size_t)(p - 1) * nn, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->beta, ctx->beta.p, (size_t)p * nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->betaSE, ctx->betaSE.p, (size_t)p * nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->stat, ctx->stat.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->pvalue, ctx->pvalue.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->deviance, ctx->deviance.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->maxCooks, ctx->maxCooks.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->normFactors, ctx->nf.p, (size_t)S * nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->mu, ctx->mu.p, (size_t)S * nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispGeneIter, ctx->dispGeneIter.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->dispIter, ctx->dispIter.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->betaIter, ctx->betaIter.p, nn)) != CD_OK) return rc;
    if ((rc = d2h(ctx, out->flags, flags, nn)) != CD_OK) return rc;
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    out->n_nonzero = (int64_t)hc[0]; out->n_gene_grid = (int64_t)hc[1];
    out->n_map_grid = (int64_t)hc[2]; out->n_beta_noconv = (int64_t)hc[3];
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]);
    ctx->timings[1] = ms;
    ctx->tm_collect();
    ctx->have_results = true;
    return CD_OK;
}

// results() (Cook's cutoff, independent filtering, BH) on n rows whose columns are in device memory on ctx's device:
// the body of cd_results_resident (the arrays of the last cd_region_test) and of cd_results_device (uploaded columns)
static int results_on_device(cd_ctx* ctx, int64_t n, int S, int p, const double* baseMean, const double* maxCooks,
                             const uint8_t* flags, const double* pvalue, double* pvalue_out, double* padj_out, double* scalars_out)
{
    cudaStream_t st = ctx->st;
    const double alpha = 0.1;
    const double cutoff = res_qf(0.99, (double)p, (double)(S - p));
    const size_t nn = (size_t)std::max<int64_t>(n, 1);
    const int C = res_chunks(n);
    for (int k = 0; k < 4; k++) CD_CUDA(ctx, ctx->res_key[k].ensure(nn));
    for (int k = 0; k < 2; k++) CD_CUDA(ctx, ctx->res_idx[k].ensure(nn));
    CD_CUDA(ctx, ctx->res_pv.ensure(nn)); CD_CUDA(ctx, ctx->res_padj.ensure(nn));
    CD_CUDA(ctx, ctx->res_bms.ensure(nn)); CD_CUDA(ctx, ctx->res_ps.ensure(nn));
    CD_CUDA(ctx, ctx->res_cnt.ensure((size_t)50 * (size_t)std::max(C, 1)));
    CD_CUDA(ctx, ctx->res_cmin.ensure((size_t)std::max(C, 1))); CD_CUDA(ctx, ctx->res_smin.ensure((size_t)std::max(C, 1)));
    CD_CUDA(ctx, ctx->res_small.ensure(2 + 50 + 50));
    CD_CUDA(ctx, ctx->res_smalld.ensure(100));
    unsigned long long* counts = ctx->res_small.p;
    unsigned long long* m_tot = ctx->res_small.p + 2;
    unsigned long long* best = ctx->res_small.p + 52;
    double* cut = ctx->res_smalld.p;
    double* theta = ctx->res_smalld.p + 50;
    unsigned long long *pkey0 = ctx->res_key[0].p, *pkey1 = ctx->res_key[1].p, *bmkey0 = ctx->res_key[2].p, *bmkey1 = ctx->res_key[3].p;
    unsigned int *idx0 = ctx->res_idx[0].p, *idx1 = ctx->res_idx[1].p;

    CD_LAUNCHN(ctx, 1, res_launch_keys(n, p, cutoff, baseMean, maxCooks, flags, pvalue, ctx->res_pv.p, ctx->res_padj.p,
                                       pkey0, bmkey0, idx0, counts, st));
    int j = 0;
    double cut_h[50], theta_h[50];
    // no rows: the host routine's values (lower = 0, upper = .95, every cut NaN)
    for (int k = 0; k < 50; k++) { cut_h[k] = NAN; theta_h[k] = (k == 49) ? .95 : 0.0 + k * ((.95 - 0.0) / 49); }
    if (n > 0) {
        size_t bytes = 0;
        CD_CUDA(ctx, cp_sort_pairs_u64(nullptr, bytes, bmkey0, bmkey1, idx0, idx1, n, st));
        CD_CUDA(ctx, ctx->res_tmp.ensure(bytes));
        CD_LAUNCHN(ctx, 1, cp_sort_pairs_u64(ctx->res_tmp.p, bytes, bmkey0, bmkey1, idx0, idx1, n, st));
        CD_LAUNCHN(ctx, 1, res_launch_cutoffs(n, bmkey1, counts, cut, theta, st));
        CD_LAUNCHN(ctx, 1, cp_sort_pairs_u64(ctx->res_tmp.p, bytes, pkey0, pkey1, idx0, idx1, n, st));
        CD_LAUNCHN(ctx, 1, res_launch_gather(n, idx1, baseMean, ctx->res_pv.p, ctx->res_bms.p, ctx->res_ps.p, st));
        CD_LAUNCHN(ctx, 3, res_launch_num_rej(n, counts, ctx->res_bms.p, ctx->res_ps.p, cut, ctx->res_cnt.p, m_tot, alpha, best, st));
        unsigned long long best_h[50];
        CD_CUDA(ctx, cudaMemcpyAsync(best_h, best, sizeof(best_h), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaMemcpyAsync(cut_h, cut, sizeof(cut_h), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaMemcpyAsync(theta_h, theta, sizeof(theta_h), cudaMemcpyDeviceToHost, st));
        CD_CUDA(ctx, cudaStreamSynchronize(st));
        double numRej[50];
        for (int k = 0; k < 50; k++) numRej[k] = (double)best_h[k];
        j = res_pick_cutoff(theta_h, numRej, 50);
        CD_LAUNCHN(ctx, 3, res_launch_bh(n, counts, ctx->res_bms.p, ctx->res_ps.p, idx1, cut, j, ctx->res_cnt.p, m_tot,
                                         ctx->res_cmin.p, ctx->res_smin.p, ctx->res_padj.p, st));
    }
    if (pvalue_out && n > 0) CD_CUDA(ctx, cudaMemcpyAsync(pvalue_out, ctx->res_pv.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    if (padj_out && n > 0) CD_CUDA(ctx, cudaMemcpyAsync(padj_out, ctx->res_padj.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CD_CUDA(ctx, cudaStreamSynchronize(st));
    if (scalars_out) {
        scalars_out[0] = cutoff; scalars_out[1] = cut_h[j]; scalars_out[2] = theta_h[j]; scalars_out[3] = (double)(j + 1);
    }
    return CD_OK;
}

int cd_results_resident(cd_ctx* ctx, double* pvalue_out, double* padj_out, double* scalars_out)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_results) return ctx->fail(CD_EINVAL, "cd_results_resident: no successful cd_region_test on this context yet");
    if (ctx->comm.active() && ctx->comm.nranks > 1)
        return ctx->fail(CD_EINVAL, "cd_results_resident: results() is global over all regions; in a sharded run gather the "
                                    "columns and call cd_results_device or cd_results_adjust");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    return results_on_device(ctx, ctx->n, ctx->des.S, ctx->des.p, ctx->g_baseMean.p + ctx->g_off, ctx->maxCooks.p,
                             ctx->g_flags.p + ctx->g_off, ctx->pvalue.p, pvalue_out, padj_out, scalars_out);
}

int cd_results_device(cd_ctx* ctx, int64_t n, int S, int p, const double* baseMean, const double* maxCooks, const uint8_t* flags,
                      const double* pvalue, double* pvalue_out, double* padj_out, double* scalars_out)
{
    if (!ctx) return CD_EINVAL;
    if (n < 0 || n > (int64_t)INT_MAX || S <= p || p < 1 || (n > 0 && (!baseMean || !pvalue)))
        return ctx->fail(CD_EINVAL, "cd_results_device: bad arguments");
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    const size_t nn = (size_t)std::max<int64_t>(n, 1), bytes = sizeof(double) * (size_t)n;
    CD_CUDA(ctx, ctx->res_in.ensure(3 * nn));                // baseMean, maxCooks, pvalue
    CD_CUDA(ctx, ctx->res_in_flags.ensure(nn));
    double *bm = ctx->res_in.p, *mc = ctx->res_in.p + nn, *pv = ctx->res_in.p + 2 * nn;
    if (n > 0) {
        CD_CUDA(ctx, cudaMemcpyAsync(bm, baseMean, bytes, cudaMemcpyHostToDevice, st));
        CD_CUDA(ctx, cudaMemcpyAsync(pv, pvalue, bytes, cudaMemcpyHostToDevice, st));
        // no maxCooks: all NaN (0xff bytes), which is never an outlier; no flags: none kept
        if (maxCooks) CD_CUDA(ctx, cudaMemcpyAsync(mc, maxCooks, bytes, cudaMemcpyHostToDevice, st));
        else CD_CUDA(ctx, cudaMemsetAsync(mc, 0xff, bytes, st));
        if (flags) CD_CUDA(ctx, cudaMemcpyAsync(ctx->res_in_flags.p, flags, (size_t)n, cudaMemcpyHostToDevice, st));
        else CD_CUDA(ctx, cudaMemsetAsync(ctx->res_in_flags.p, 0, (size_t)n, st));
    }
    return results_on_device(ctx, n, S, p, bm, mc, ctx->res_in_flags.p, pv, pvalue_out, padj_out, scalars_out);
}

int cd_get_dims(const cd_ctx* ctx, int64_t* n, int* S, int* p, int64_t* R)
{
    if (!ctx) return CD_EINVAL;
    if (n) *n = ctx->n;
    if (S) *S = ctx->have_design ? ctx->des.S : 0;
    if (p) *p = ctx->have_design ? ctx->des.p : 0;
    if (R) *R = ctx->R;
    return CD_OK;
}

int64_t cd_launch_count(const cd_ctx* ctx) { return ctx ? ctx->launches : 0; }

int cd_timer_start(cd_ctx* ctx)
{
    if (!ctx) return CD_EINVAL;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, cudaEventRecord(ctx->ev_user[0], ctx->st));
    return CD_OK;
}

int cd_timer_stop(cd_ctx* ctx, double* ms_out)
{
    if (!ctx || !ms_out) return CD_EINVAL;
    CD_CUDA(ctx, cudaEventRecord(ctx->ev_user[1], ctx->st));
    CD_CUDA(ctx, cudaEventSynchronize(ctx->ev_user[1]));
    float ms = 0;
    CD_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev_user[0], ctx->ev_user[1]));
    *ms_out = ms;
    return CD_OK;
}

int cd_measure_fp64_peak(cd_ctx* ctx, double* tflops_out)
{
    if (!ctx || !tflops_out) return CD_EINVAL;
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    CD_CUDA(ctx, ctx->scal.ensure(128));
    const int blocks = 148 * 8, threads = 256, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CD_CUDA(ctx, cudaEventRecord(ctx->ev_user[0], ctx->st));
        dfma_peak_kernel<<<blocks, threads, 0, ctx->st>>>(iters, 1.0000001, ctx->scal.p + 100);
        ctx->launches++;
        CD_CUDA(ctx, cudaEventRecord(ctx->ev_user[1], ctx->st));
        CD_CUDA(ctx, cudaEventSynchronize(ctx->ev_user[1]));
        float ms = 0;
        CD_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev_user[0], ctx->ev_user[1]));
        const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *tflops_out = best;
    return CD_OK;
}

int cd_device_buffers(cd_ctx* ctx, const int32_t** K_dev, const double** fullmean_dev)
{
    if (!ctx) return CD_EINVAL;
    if (!ctx->have_agg) return ctx->fail(CD_EINVAL, "cd_device_buffers: nothing aggregated yet");
    if (K_dev) *K_dev = ctx->K.p;
    if (fullmean_dev) *fullmean_dev = ctx->FM.p;
    return CD_OK;
}

int cd_last_search_counts(const cd_ctx* ctx, int* n_calls, int64_t evaluations[16], int design_columns[16], int64_t regions[16])
{
    if (!ctx || !n_calls) return CD_EINVAL;
    *n_calls = ctx->n_eval_calls;
    for (int k = 0; k < 16; k++) {
        if (evaluations) evaluations[k] = k < ctx->n_eval_calls ? (int64_t)ctx->eval_counts_host[k] : 0;
        if (design_columns) design_columns[k] = k < ctx->n_eval_calls ? ctx->eval_call_p[k] : 0;
        if (regions) regions[k] = k < ctx->n_eval_calls ? ctx->eval_call_regions[k] : 0;
    }
    return CD_OK;
}

int cd_last_rendezvous(const cd_ctx* ctx, double* trend_passes, double* wait_cycles_peers, double* wait_cycles_self,
                       double* wait_cycles_first_pass)
{
    if (!ctx) return CD_EINVAL;
    if (trend_passes) *trend_passes = ctx->trend_passes;
    if (wait_cycles_peers) *wait_cycles_peers = (double)ctx->wait_host[0];
    if (wait_cycles_self) *wait_cycles_self = (double)ctx->wait_host[1];
    if (wait_cycles_first_pass) *wait_cycles_first_pass = (double)ctx->wait_host[2];
    return CD_OK;
}

int cd_ihw_apply_device(cd_ctx* ctx, int64_t n, const double* avDist, const double* pvalue, int ngroups, const double* minLogDist,
                        const double* maxLogDist, const double* avWeights, int32_t* group_out, double* weight_out,
                        double* weighted_pvalue_out, double* weighted_padj_out)
{
    if (!ctx) return CD_EINVAL;
    if (n < 0 || ngroups < 1 || !minLogDist || !maxLogDist || !avWeights || (n > 0 && !pvalue))
        return ctx->fail(CD_EINVAL, "cd_ihw_apply_device: bad arguments");
    if (!avDist && (!ctx->avDist.p || n != ctx->n || !ctx->have_agg))
        return ctx->fail(CD_EINVAL, "cd_ihw_apply_device: no avDist given and none of %lld regions left on the device by cd_assemble",
                         (long long)n);
    CD_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->st;
    DevBuf<double> in;                                   // pvalue, then avDist when it comes from the host
    CD_CUDA(ctx, in.ensure((size_t)std::max<int64_t>(2 * n, 1)));
    if (n > 0) {
        CD_CUDA(ctx, cudaMemcpyAsync(in.p, pvalue, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
        if (avDist) CD_CUDA(ctx, cudaMemcpyAsync(in.p + n, avDist, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    bool bad_breaks = false;
    const cudaError_t e = ihw_apply_device(n, avDist ? in.p + n : ctx->avDist.p, in.p, ngroups, minLogDist, maxLogDist, avWeights,
                                           group_out, weight_out, weighted_pvalue_out, weighted_padj_out, &bad_breaks, st);
    ctx->launches += (n > 0 && e == cudaSuccess) ? (weighted_padj_out ? 4 : 2) : 0;
    if (bad_breaks) return ctx->fail(CD_EINVAL, "cd_ihw_apply_device: a break is NaN or 'breaks' are not unique");
    if (e != cudaSuccess) return ctx->fail(CD_ECUDA, "cd_ihw_apply_device: %s", cudaGetErrorString(e));
    return CD_OK;
}

int cd_last_timings(const cd_ctx* ctx, double out_ms[8])
{
    if (!ctx || !out_ms) return CD_EINVAL;
    for (int k = 0; k < 8; k++) out_ms[k] = ctx->timings[k];
    return CD_OK;
}

}  // extern "C"
