// engine.cu -- host side of libpqb200.so: the C ABI of include/pqb200.h over the fused
// sm_100a suite kernel (suite_kernel.cuh).  Plain CUDA runtime; no torch, no CPU fallback:
// every compute entry point fails loudly when there is no device.
//
// Device layout: every plane (4 inputs, 21 outputs) is "tiled"
//   [symbol block of 32][bar][32 symbols]                          (suite_kernel.cuh, DESIGN.md 3)
// Host staging (pinned) and everything that crosses the ABI is row-major Arrow-style
// [symbol][pitch] f64 + LSB-first validity bitmaps; pack_kernel / unpack_kernel convert on the
// device, chunk by chunk, on the way in and out.
#include "../../include/pqb200.h"
#include "../../include/pqb200_polars_plugin.h"   // the Arrow C Data Interface structs
#include "suite_kernel.cuh"
#include "candles.cuh"
#include "longrows.cuh"
#include "windows.cuh"

#include <algorithm>
#include <atomic>
#include <map>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <memory>
#include <vector>

using namespace pqb;

// ---------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            int code__ = (e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver)         \
                             ? PQB_ERR_NO_DEVICE : PQB_ERR_CUDA;                                  \
            return fail(code__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
        }                                                                                         \
    } while (0)

extern "C" const char *pqb_last_error(void) { return g_err.c_str(); }
extern "C" int pqb_abi_version(void) { return PQB_ABI_VERSION; }

extern "C" int pqb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int good = 0;
    for (int d = 0; d < n; ++d) {
        cudaDeviceProp pr;
        if (cudaGetDeviceProperties(&pr, d) == cudaSuccess && pr.major == 10) ++good;
    }
    return good;
}

extern "C" void pqb_suite_params_default(pqb_suite_params *p) {
    if (!p) return;
    p->indicators = PQB_IND_ALL;
    p->sma_period = 30; p->ema_period = 30; p->tema_period = 30; p->trima_period = 30;
    p->bbands_period = 20; p->bbands_nbdevup = 2.0; p->bbands_nbdevdn = 2.0;
    p->macd_fast = 12; p->macd_slow = 26; p->macd_signal = 9;
    p->rsi_period = 14; p->atr_period = 14; p->natr_period = 14;
    p->kdj_fastk = 9; p->kdj_slowk = 3; p->kdj_slowd = 3;
    p->willr_period = 14; p->midprice_period = 14;
    p->midpoint_period = 14; p->adosc_fast = 3; p->adosc_slow = 10; p->mom_period = 10; p->roc_period = 10;
    p->cmo_period = 14; p->mfi_period = 14; p->cci_period = 14; p->dm_period = 14;
    p->trix_period = 30; p->ultosc_period1 = 7; p->ultosc_period2 = 14; p->ultosc_period3 = 28; p->aroon_period = 14;
    p->donchian_period = 20;
}

// ---------------------------------------------------------------------------------------
// engine / panel objects
// ---------------------------------------------------------------------------------------
static constexpr int kMaxSmem = 227 * 1024;      // opt-in dynamic shared memory per CTA on sm_100
static constexpr int kSmemThreeCtas = 75 * 1024; // (228 KB per SM - 1 KB reserved per CTA) / 3
static constexpr int kFixedSmem = NS * STAGE_BYTES + 2 * NS * 8;   // TMA stages (+ validity words) + mbarriers

struct pqb_engine {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // compute
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaStream_t aux = nullptr;          // the compact tail launch of a small panel runs beside the main launch (launch_suite)
    cudaStream_t side = nullptr;         // per-block null dispatch: the null-aware launch beside the plain one (which may use `aux` itself)
    cudaEvent_t ev_side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_pre = nullptr;
    void *flush_buf = nullptr;
    size_t flush_bytes = 0;
    std::mutex mu;                       // guards the single-column scratch panel
    pqb_panel *scratch = nullptr;
    int64_t scratch_bars = 0;
    // a few one-symbol scratch panels of the lengths seen lately (a frame usually holds columns of one or two lengths; the single-
    // column entry points used to re-create the scratch -- 4 + 44 planes -- whenever the length changed)
    std::vector<std::pair<int64_t, pqb_panel *>> scratch_lru;
    pqb_candles *cscratch = nullptr;     // single-column scratch of the candle engine (candles_host.inc)
    int64_t cscratch_bars = 0;
    // pinned staging planes of destroyed panels, kept for the next panel of the same shape: page-locking is the
    // expensive part of creating a panel (measured: 0.48 s of a 0.9 s WidePanel.suite() call on 2,000 x 2,520)
    // panels hold a pointer to their engine: pqb_engine_destroy() with panels still alive (a garbage collector finalising
    // objects in any order) only marks the engine, and the last panel to go frees it
    int live_panels = 0;
    bool destroy_requested = false;
    std::mutex pool_mu;                  // guards live_panels / destroy_requested / the pool
    std::multimap<size_t, void *> host_pool;
    size_t host_pool_bytes = 0, host_pool_cap = 4ull << 30;
    // ... and their device planes: cudaMalloc / cudaFree of ~60 buffers were 40 ms of a 130 ms WidePanel.suite() call on
    // 2,000 x 2,520 (cudaFree synchronises the device); PQB_DEV_POOL_MB, default 4096
    std::multimap<size_t, void *> dev_pool;
    size_t dev_pool_bytes = 0, dev_pool_cap = 4ull << 30;
};

// CUDA events that are destroyed on every way out of a function (the CU() macro returns early)
struct Events {
    std::vector<cudaEvent_t> ev;
    explicit Events(size_t n) : ev(n, nullptr) {}
    ~Events() { for (cudaEvent_t x : ev) if (x) cudaEventDestroy(x); }
    cudaEvent_t &operator[](size_t i) { return ev[i]; }
    cudaError_t create(unsigned flags = cudaEventDefault) {
        for (cudaEvent_t &x : ev) { const cudaError_t ce = cudaEventCreateWithFlags(&x, flags); if (ce != cudaSuccess) return ce; }
        return cudaSuccess;
    }
};

// page-locked host memory placed next to the engine's GPU (columns_host.inc: the calling thread runs on the GPU-local
// CPUs while the driver allocates and pins the pages)
static cudaError_t host_alloc_local(pqb_engine *e, void **out, size_t bytes);
static cudaError_t host_take(pqb_engine *e, void **out, size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        auto it = e->host_pool.find(bytes);
        if (it != e->host_pool.end()) {
            *out = it->second;
            e->host_pool.erase(it);
            e->host_pool_bytes -= bytes;
            return cudaSuccess;
        }
    }
    cudaError_t ce = host_alloc_local(e, out, bytes);
    if (ce == cudaSuccess) return ce;
    cudaGetLastError();
    {                                                   // out of pinned memory: give the pool back and try once more
        std::lock_guard<std::mutex> lk(e->pool_mu);
        for (auto &kv : e->host_pool) cudaFreeHost(kv.second);
        e->host_pool.clear();
        e->host_pool_bytes = 0;
    }
    return host_alloc_local(e, out, bytes);
}

static void host_give(pqb_engine *e, void *ptr, size_t bytes) {
    if (!ptr) return;
    if (e) {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        if (e->host_pool_bytes + bytes <= e->host_pool_cap) {
            e->host_pool.emplace(bytes, ptr);
            e->host_pool_bytes += bytes;
            return;
        }
    }
    cudaFreeHost(ptr);
}

static cudaError_t dev_take(pqb_engine *e, void **out, size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        auto it = e->dev_pool.find(bytes);
        if (it != e->dev_pool.end()) {
            *out = it->second;
            e->dev_pool.erase(it);
            e->dev_pool_bytes -= bytes;
            return cudaSuccess;
        }
    }
    cudaError_t ce = cudaMalloc(out, bytes);
    if (ce == cudaSuccess) return ce;
    cudaGetLastError();
    {                                                   // out of device memory: give the pool back and try once more
        std::lock_guard<std::mutex> lk(e->pool_mu);
        for (auto &kv : e->dev_pool) cudaFree(kv.second);
        e->dev_pool.clear();
        e->dev_pool_bytes = 0;
    }
    return cudaMalloc(out, bytes);
}

// (the caller has synchronised the streams that used the buffer: a pooled buffer is handed out again without a device sync)
static void dev_give(pqb_engine *e, void *ptr, size_t bytes) {
    if (!ptr) return;
    if (e) {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        if (e->dev_pool_bytes + bytes <= e->dev_pool_cap) {
            e->dev_pool.emplace(bytes, ptr);
            e->dev_pool_bytes += bytes;
            return;
        }
    }
    cudaFree(ptr);
}

struct pqb_panel;
static void export_cache_drop(pqb_panel *p);

struct pqb_panel {
    // the panel itself holds one reference, every outstanding Arrow export (pqb_panel_export_arrow) another: the
    // pinned result planes an export aliases live until the last of them is released
    std::atomic<int> refs{1};
    std::mutex export_mu;                // the vectors of a released Arrow export, kept for the next one (columns_host.inc)
    void *export_cache_a = nullptr, *export_cache_s = nullptr;
    pqb_engine *e = nullptr;
    int64_t n_symbols = 0, n_bars = 0, pitch = 0, words_per_row = 0;
    int64_t n_blocks = 0, bars_padded = 0;   // tiled geometry
    size_t plane_doubles = 0;            // n_blocks * bars_padded * 32
    uint32_t fields_mask = 0;
    uint64_t outputs_mask = 0;
    double *d_in[PQB_N_FIELDS] = {};     // tiled
    double *d_out[PQB_N_OUTPUTS] = {};   // tiled
    uint32_t *d_bits[PQB_N_OUTPUTS] = {};// row-major bitmaps
    int *d_start = nullptr;
    bool starts_nonzero = false;
    // pinned row-major staging
    double *h_in[PQB_N_FIELDS] = {};
    double *h_out[PQB_N_OUTPUTS] = {};
    uint32_t *h_bits[PQB_N_OUTPUTS] = {};
    std::vector<int32_t> h_start;
    bool staging = false;
    // device row-major transfer buffers: 2 x chunk for inputs and outputs (double-buffered)
    int64_t chunk_symbols = 0;
    double *d_xin[2] = {};               // [n_fields_alloc][chunk][pitch]
    double *d_xout[2] = {};              // [n_outputs_alloc][chunk][pitch]
    int n_in_alloc = 0, n_out_alloc = 0;
    int in_slot[PQB_N_FIELDS] = {}, out_slot[PQB_N_OUTPUTS] = {};
    cudaEvent_t ev_packed[2] = {}, ev_d2h[2] = {};
    int last_launches = 0;               // kernels launched by the most recent run / run_host
    // null-aware mode (allocated on first use)
    std::vector<int32_t> h_start_explicit;              // pqb_panel_set_starts
    std::vector<int32_t> h_lead[PQB_N_FIELDS];          // leading nulls seen by pqb_panel_set_column (-1: none given)
    std::vector<uint32_t> h_vin[PQB_N_FIELDS];          // row-major input validity bitmaps (empty: all valid)
    std::vector<uint8_t> h_flags;                       // per symbol: bit f = field f has an interior/trailing null
    bool nulls_mode = false;                            // some symbol block needs the null-aware kernel (prepare_nulls)
    std::vector<uint8_t> h_blk_null;                    // per symbol block: 1 = interior / trailing nulls or fields starting at different rows
    int64_t n_null_blocks = 0;
    std::vector<int> h_blist;                           // [2][n_blocks]: plain blocks, then null blocks, of the ranges launched so far
    int *d_blist = nullptr;
    uint32_t *d_vin[PQB_N_FIELDS] = {};                 // row-major bitmaps on the device
    uint32_t *d_vmask = nullptr;                        // tiled [block][bar][4]
    uint32_t *d_ovm[PQB_N_OUTPUTS] = {};                // tiled [block][bar] per output
    uint8_t *d_flags = nullptr;
    // symbol compaction (prepare_nulls / launch_suite): the flagged symbols of a device-resident panel copied into blocks of
    // their own.  x slot i holds symbol h_symmap[i].
    bool compact = false;                               // the structures below describe the panel's current columns
    int64_t n_x = 0, n_xblocks = 0, x_cap_blocks = 0;   // flagged symbols, their blocks, blocks allocated
    std::vector<int32_t> h_symmap, h_xstart;            // x slot -> symbol (-1: empty); explicit starts of the slots
    std::vector<uint8_t> h_xflags;
    std::vector<int32_t> h_start_c;                     // starts by the plain rule for EVERY symbol (the plain kernel runs all blocks)
    int *d_symmap = nullptr, *d_xstart = nullptr, *d_start_c = nullptr;
    uint8_t *d_xflags = nullptr;
    double *x_in[PQB_N_FIELDS] = {}, *x_out[PQB_N_OUTPUTS] = {};
    uint32_t *x_vmask = nullptr, *x_ovm[PQB_N_OUTPUTS] = {};
    // crossover signals (signals_host.inc): row-major int8 planes, allocated on first use
    int8_t *d_sig = nullptr, *h_sig = nullptr;
    bool inputs_resident = false;        // the tiled input planes hold the panel (upload / run_host / fill_synthetic)
    bool retained = false;               // registered with the engine (engine_retain)
    double *d_info = nullptr;            // last-row reductions (info_host.inc): [PQB_N_INFO][n_symbols] + validity bytes
    uint8_t *d_info_valid = nullptr;
};

static int set_dev(const pqb_engine *e) {
    CU(cudaSetDevice(e->device));
    return PQB_OK;
}

static void engine_free(pqb_engine *e);

extern "C" int pqb_engine_create(int device, pqb_engine **out) {
    if (!out) return fail(PQB_ERR_INVALID, "pqb_engine_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(PQB_ERR_NO_DEVICE, "no CUDA device (%s): the engine has no CPU fallback",
                    ce == cudaSuccess ? "device count 0" : cudaGetErrorString(ce));
    }
    if (device < 0 || device >= n) return fail(PQB_ERR_INVALID, "device %d out of range [0,%d)", device, n);
    cudaDeviceProp pr;
    CU(cudaGetDeviceProperties(&pr, device));
    if (pr.major != 10)
        return fail(PQB_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    pr.major, pr.minor);
    pqb_engine *e = new pqb_engine();
    std::unique_ptr<pqb_engine, void (*)(pqb_engine *)> guard(e, engine_free);       // (freed on every early return below)
    e->device = device;
    e->sm_count = pr.multiProcessorCount;
    if (const char *hp = getenv("PQB_HOST_POOL_MB")) e->host_pool_cap = (size_t)std::max(0, atoi(hp)) << 20;   // 0: no pooling
    if (const char *dp = getenv("PQB_DEV_POOL_MB")) e->dev_pool_cap = (size_t)std::max(0, atoi(dp)) << 20;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&e->h2d, cudaStreamNonBlocking));
    {   // the second stream carries the short side launches that must START beside a grid-filling main launch (compact tail CTAs,
        // the null-aware kernel over compacted blocks): highest priority, so that their CTAs are placed first
        int least = 0, greatest = 0;
        CU(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CU(cudaStreamCreateWithPriority(&e->aux, cudaStreamNonBlocking, greatest));
        CU(cudaStreamCreateWithPriority(&e->side, cudaStreamNonBlocking, greatest));
    }
    CU(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_side, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_pre, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&e->d2h, cudaStreamNonBlocking));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, true, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
    CU(cudaFuncSetAttribute(suite_fused_kernel<false, false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    guard.release();
    *out = e;
    return PQB_OK;
}

static void engine_free(pqb_engine *e) {
    cudaSetDevice(e->device);
    for (auto &kv : e->host_pool) cudaFreeHost(kv.second);
    for (auto &kv : e->dev_pool) cudaFree(kv.second);
    if (e->flush_buf) cudaFree(e->flush_buf);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->h2d) cudaStreamDestroy(e->h2d);
    if (e->aux) cudaStreamDestroy(e->aux);
    if (e->side) cudaStreamDestroy(e->side);
    if (e->ev_side) cudaEventDestroy(e->ev_side);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->ev_pre) cudaEventDestroy(e->ev_pre);
    if (e->d2h) cudaStreamDestroy(e->d2h);
    delete e;
}

extern "C" void pqb_engine_destroy(pqb_engine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->scratch) { pqb_panel_destroy(e->scratch); e->scratch = nullptr; }
    for (auto &kv : e->scratch_lru) pqb_panel_destroy(kv.second);
    e->scratch_lru.clear();
    if (e->cscratch) { pqb_candles_destroy(e->cscratch); e->cscratch = nullptr; }
    {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        if (e->live_panels > 0) { e->destroy_requested = true; return; }      // the last panel frees the engine
    }
    engine_free(e);
}

// a panel (suite or candle) registers with / leaves its engine
static void engine_retain(pqb_engine *e) {
    std::lock_guard<std::mutex> lk(e->pool_mu);
    ++e->live_panels;
}
static void engine_release(pqb_engine *e) {
    bool last;
    {
        std::lock_guard<std::mutex> lk(e->pool_mu);
        last = --e->live_panels == 0 && e->destroy_requested;
    }
    if (last) engine_free(e);
}

extern "C" int pqb_panel_create(pqb_engine *e, int64_t n_symbols, int64_t n_bars, uint32_t fields_mask,
                                uint64_t outputs_mask, int host_staging, pqb_panel **out) {
    if (!e || !out) return fail(PQB_ERR_INVALID, "pqb_panel_create: NULL argument");
    *out = nullptr;
    if (n_symbols <= 0 || n_bars <= 0 || n_symbols > (1ll << 30) || n_bars > (1ll << 30))
        return fail(PQB_ERR_INVALID, "pqb_panel_create: bad shape %lld x %lld", (long long)n_symbols, (long long)n_bars);
    if (fields_mask == 0 || fields_mask >= (1u << PQB_N_FIELDS) || outputs_mask >= (1ull << PQB_N_OUTPUTS))
        return fail(PQB_ERR_INVALID, "pqb_panel_create: bad masks");
    int rc = set_dev(e);
    if (rc) return rc;
    pqb_panel *p = new pqb_panel();
    p->e = e;
    engine_retain(e);
    p->retained = true;
    p->n_symbols = n_symbols;
    p->n_bars = n_bars;
    p->pitch = (n_bars + 15) / 16 * 16;
    p->words_per_row = (n_bars + 31) / 32;
    p->n_blocks = (n_symbols + SYM - 1) / SYM;
    p->bars_padded = (n_bars + SB - 1) / SB * SB;
    p->plane_doubles = (size_t)p->n_blocks * p->bars_padded * SYM;
    p->fields_mask = fields_mask;
    p->outputs_mask = outputs_mask;
    p->staging = host_staging != 0;
    const size_t hplane = (size_t)n_symbols * p->pitch * sizeof(double);
    const size_t dplane = p->plane_doubles * sizeof(double);
    const size_t bplane = (size_t)n_symbols * p->words_per_row * sizeof(uint32_t);
    auto bail = [&](cudaError_t ce, const char *what) {
        const int code = ce == cudaErrorMemoryAllocation ? PQB_ERR_ALLOC : PQB_ERR_CUDA;
        fail(code, "pqb_panel_create: %s: %s", what, cudaGetErrorString(ce));
        cudaGetLastError();
        pqb_panel_destroy(p);
        return code;
    };
    cudaError_t ce;
    for (int f = 0; f < PQB_N_FIELDS; ++f) {
        if (!(fields_mask >> f & 1)) continue;
        if ((ce = dev_take(e, (void **)&p->d_in[f], dplane)) != cudaSuccess) return bail(ce, "cudaMalloc(field)");
        if ((ce = cudaMemsetAsync(p->d_in[f], 0, dplane, e->stream)) != cudaSuccess) return bail(ce, "memset");
        p->in_slot[f] = p->n_in_alloc++;
        if (p->staging) {
            if ((ce = host_take(e, (void **)&p->h_in[f], hplane)) != cudaSuccess) return bail(ce, "cudaMallocHost(field)");
            if (host_staging != 2) memset(p->h_in[f], 0, hplane);
        }
    }
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) {
        if (!(outputs_mask >> k & 1)) continue;
        if ((ce = dev_take(e, (void **)&p->d_out[k], dplane)) != cudaSuccess) return bail(ce, "cudaMalloc(output)");
        if ((ce = dev_take(e, (void **)&p->d_bits[k], bplane)) != cudaSuccess) return bail(ce, "cudaMalloc(validity)");
        p->out_slot[k] = p->n_out_alloc++;
        if (p->staging) {
            if ((ce = host_take(e, (void **)&p->h_out[k], hplane)) != cudaSuccess) return bail(ce, "cudaMallocHost(output)");
            if ((ce = host_take(e, (void **)&p->h_bits[k], bplane)) != cudaSuccess) return bail(ce, "cudaMallocHost(validity)");
        }
    }
    if (p->staging) {
        // transfer chunk: whole symbol blocks, at most ~32 MB per plane
        int64_t cs = (32ll << 20) / (p->pitch * (int64_t)sizeof(double));
        cs = std::max<int64_t>(SYM, cs / SYM * SYM);
        cs = std::min<int64_t>(cs, p->n_blocks * SYM);
        p->chunk_symbols = cs;
        const size_t cplane = (size_t)cs * p->pitch * sizeof(double);
        for (int b = 0; b < 2; ++b) {
            if ((ce = dev_take(e, (void **)&p->d_xin[b], cplane * p->n_in_alloc)) != cudaSuccess) return bail(ce, "cudaMalloc(xfer in)");
            if (p->n_out_alloc &&
                (ce = dev_take(e, (void **)&p->d_xout[b], cplane * p->n_out_alloc)) != cudaSuccess) return bail(ce, "cudaMalloc(xfer out)");
            if ((ce = cudaEventCreateWithFlags(&p->ev_packed[b], cudaEventDisableTiming)) != cudaSuccess) return bail(ce, "event");
            if ((ce = cudaEventCreateWithFlags(&p->ev_d2h[b], cudaEventDisableTiming)) != cudaSuccess) return bail(ce, "event");
        }
    }
    if ((ce = cudaMalloc(&p->d_start, (size_t)p->n_blocks * SYM * sizeof(int))) != cudaSuccess) return bail(ce, "cudaMalloc(start)");
    if ((ce = cudaMemsetAsync(p->d_start, 0, (size_t)p->n_blocks * SYM * sizeof(int), e->stream)) != cudaSuccess) return bail(ce, "memset");
    p->h_start.assign((size_t)n_symbols, 0);
    p->h_start_explicit.assign((size_t)n_symbols, 0);
    for (auto &v : p->h_lead) v.assign((size_t)n_symbols, -1);
    p->h_flags.assign((size_t)n_symbols, 0);
    p->h_blk_null.assign((size_t)p->n_blocks, 0);
    if ((ce = cudaStreamSynchronize(e->stream)) != cudaSuccess) return bail(ce, "sync");
    *out = p;
    return PQB_OK;
}

extern "C" void pqb_panel_destroy(pqb_panel *p) {
    if (!p) return;
    if (p->refs.fetch_sub(1) > 1) return;            // exports still alias the result planes: the last release frees
    export_cache_drop(p);
    if (p->e) cudaSetDevice(p->e->device);
    // the big planes go back to the engine's device pool (dev_give): nothing may still be running on them
    if (p->e) {
        cudaStreamSynchronize(p->e->stream);
        cudaStreamSynchronize(p->e->h2d);
        cudaStreamSynchronize(p->e->d2h);
    }
    {
        const size_t dplane_ = p->plane_doubles * sizeof(double);
        const size_t bplane_ = (size_t)p->n_symbols * p->words_per_row * sizeof(uint32_t);
        const size_t cplane_ = (size_t)p->chunk_symbols * p->pitch * sizeof(double);
        for (auto &q : p->d_in) dev_give(p->e, q, dplane_);
        for (auto &q : p->d_out) dev_give(p->e, q, dplane_);
        for (auto &q : p->d_bits) dev_give(p->e, q, bplane_);
        for (auto &q : p->d_xin) dev_give(p->e, q, cplane_ * p->n_in_alloc);
        for (auto &q : p->d_xout) dev_give(p->e, q, cplane_ * p->n_out_alloc);
    }
    if (p->d_start) cudaFree(p->d_start);
    for (auto &q : p->d_vin) if (q) cudaFree(q);
    for (auto &q : p->d_ovm) if (q) cudaFree(q);
    if (p->d_vmask) cudaFree(p->d_vmask);
    if (p->d_flags) cudaFree(p->d_flags);
    if (p->d_blist) cudaFree(p->d_blist);
    for (auto &q : p->x_in) if (q) cudaFree(q);
    for (auto &q : p->x_out) if (q) cudaFree(q);
    for (auto &q : p->x_ovm) if (q) cudaFree(q);
    if (p->x_vmask) cudaFree(p->x_vmask);
    if (p->d_symmap) cudaFree(p->d_symmap);
    if (p->d_xstart) cudaFree(p->d_xstart);
    if (p->d_start_c) cudaFree(p->d_start_c);
    if (p->d_xflags) cudaFree(p->d_xflags);
    if (p->d_sig) cudaFree(p->d_sig);
    if (p->d_info) cudaFree(p->d_info);
    if (p->d_info_valid) cudaFree(p->d_info_valid);
    if (p->h_sig) cudaFreeHost(p->h_sig);
    const size_t hplane = (size_t)p->n_symbols * p->pitch * sizeof(double);
    const size_t bplane = (size_t)p->n_symbols * p->words_per_row * sizeof(uint32_t);
    for (auto &q : p->h_in) host_give(p->e, q, hplane);
    for (auto &q : p->h_out) host_give(p->e, q, hplane);
    for (auto &q : p->h_bits) host_give(p->e, q, bplane);
    for (auto &ev : p->ev_packed) if (ev) cudaEventDestroy(ev);
    for (auto &ev : p->ev_d2h) if (ev) cudaEventDestroy(ev);
    pqb_engine *e = p->retained ? p->e : nullptr;
    delete p;
    if (e) engine_release(e);
}

extern "C" int64_t pqb_panel_pitch(const pqb_panel *p) { return p ? p->pitch : 0; }
extern "C" int64_t pqb_panel_validity_pitch(const pqb_panel *p) { return p ? p->words_per_row * 4 : 0; }
extern "C" int pqb_panel_tiled_shape(const pqb_panel *p, int64_t *n_blocks, int64_t *bars_padded) {
    if (!p) return fail(PQB_ERR_INVALID, "pqb_panel_tiled_shape: NULL");
    if (n_blocks) *n_blocks = p->n_blocks;
    if (bars_padded) *bars_padded = p->bars_padded;
    return PQB_OK;
}
extern "C" double *pqb_panel_host_field(pqb_panel *p, int f) {
    return (p && f >= 0 && f < PQB_N_FIELDS) ? p->h_in[f] : nullptr;
}
extern "C" const double *pqb_panel_host_output(pqb_panel *p, int k) {
    return (p && k >= 0 && k < PQB_N_OUTPUTS) ? p->h_out[k] : nullptr;
}
extern "C" const uint8_t *pqb_panel_host_validity(pqb_panel *p, int k) {
    return (p && k >= 0 && k < PQB_N_OUTPUTS) ? reinterpret_cast<const uint8_t *>(p->h_bits[k]) : nullptr;
}
extern "C" const double *pqb_panel_device_field(const pqb_panel *p, int f) {
    return (p && f >= 0 && f < PQB_N_FIELDS) ? p->d_in[f] : nullptr;
}
extern "C" const double *pqb_panel_device_output(const pqb_panel *p, int k) {
    return (p && k >= 0 && k < PQB_N_OUTPUTS) ? p->d_out[k] : nullptr;
}
extern "C" const uint8_t *pqb_panel_device_validity(const pqb_panel *p, int k) {
    return (p && k >= 0 && k < PQB_N_OUTPUTS) ? reinterpret_cast<const uint8_t *>(p->d_bits[k]) : nullptr;
}

static inline bool bit_at(const uint8_t *bm, int64_t i) { return (bm[i >> 3] >> (i & 7)) & 1; }
// (columns_host.inc)
static void ensure_vin(pqb_panel *p, int field);
static int stage_column(pqb_panel *p, int64_t symbol, int field, const void *values, char fmt, const uint8_t *validity,
                        int64_t offset, int64_t len);

extern "C" int pqb_panel_set_column(pqb_panel *p, int64_t symbol, int field, const double *values,
                                    const uint8_t *validity, int64_t offset, int64_t len) {
    if (!p || !values) return fail(PQB_ERR_INVALID, "pqb_panel_set_column: NULL argument");
    if (!p->staging) return fail(PQB_ERR_INVALID, "pqb_panel_set_column: panel has no host staging");
    if (symbol < 0 || symbol >= p->n_symbols || field < 0 || field >= PQB_N_FIELDS || !p->h_in[field])
        return fail(PQB_ERR_INVALID, "pqb_panel_set_column: bad symbol/field");
    if (len != p->n_bars || offset < 0)
        return fail(PQB_ERR_INVALID, "pqb_panel_set_column: len %lld != n_bars %lld", (long long)len, (long long)p->n_bars);
    if (validity) ensure_vin(p, field);
    return stage_column(p, symbol, field, values, 'g', validity, offset, len);
}

extern "C" int pqb_panel_clear_validity(pqb_panel *p, int field) {
    if (!p || field >= PQB_N_FIELDS) return fail(PQB_ERR_INVALID, "pqb_panel_clear_validity: bad argument");
    for (int f = 0; f < PQB_N_FIELDS; ++f) {
        if (field >= 0 && f != field) continue;
        std::fill(p->h_lead[f].begin(), p->h_lead[f].end(), -1);
        p->h_vin[f].clear();
        for (auto &fl : p->h_flags) fl &= (uint8_t)~(1u << f);
    }
    return PQB_OK;
}

extern "C" int pqb_panel_set_starts(pqb_panel *p, const int32_t *starts) {
    if (!p || !starts) return fail(PQB_ERR_INVALID, "pqb_panel_set_starts: NULL argument");
    for (int64_t s = 0; s < p->n_symbols; ++s) {
        if (starts[s] < 0) return fail(PQB_ERR_INVALID, "pqb_panel_set_starts: negative start");
        p->h_start_explicit[(size_t)s] = (int32_t)std::min<int64_t>(starts[s], p->n_bars);
    }
    return PQB_OK;
}

// Symbol compaction (whole-panel prepare only, i.e. the device-resident path).  Per-block dispatch sends every block that
// holds ONE flagged symbol through the null-aware kernel, whose walk is ~3x longer per bar than the plain kernel's and whose
// CTAs are twice as heavy: 500 halted symbols spread over a 50,000-symbol panel flag 430 of its 1,563 blocks.  When the
// flagged symbols are few, they are copied into blocks of their own instead (compact_kernel<true>), the null-aware kernel
// walks those ceil(n / 32) blocks on the engine's second stream, the plain kernel runs EVERY original block beside it (the
// flagged symbols' lanes compute on benign values and are overwritten afterwards: compact_kernel<false>, unpack of the
// compacted validity words), and nothing else changes -- same kernels, same arithmetic, same bits.
static bool compaction_enabled() {
    static const bool v = !getenv("PQB_COMPACT_NULLS") || atoi(getenv("PQB_COMPACT_NULLS")) != 0;
    return v;
}
static int prepare_compaction(pqb_panel *p, cudaStream_t st) {
    if (!compaction_enabled() || !p->nulls_mode) return PQB_OK;
    // flagged symbols: an interior / trailing null, or fields starting at different rows
    std::vector<int32_t> &map = p->h_symmap;
    map.clear();
    p->h_start_c.assign((size_t)p->n_symbols, 0);
    for (int64_t s = 0; s < p->n_symbols; ++s) {
        bool flagged = p->h_flags[(size_t)s] != 0;
        int32_t lead = -2, a = p->h_start_explicit[(size_t)s];
        for (int f = 0; f < PQB_N_FIELDS; ++f) {
            if (!p->d_in[f] || p->h_lead[f][(size_t)s] < 0) continue;
            if (lead == -2) lead = p->h_lead[f][(size_t)s];
            else if (lead != p->h_lead[f][(size_t)s]) flagged = true;
            a = std::max(a, p->h_lead[f][(size_t)s]);
        }
        p->h_start_c[(size_t)s] = a;
        if (flagged) map.push_back((int32_t)s);
    }
    const int64_t n_x = (int64_t)map.size(), n_xb = (n_x + SYM - 1) / SYM;
    // worth it only while the compacted blocks are few next to the blocks they replace and next to the SMs
    // worth it while the compacted blocks are few next to the blocks they replace, fit the GPU beside the plain launch (two
    // null-aware CTAs per SM) and the write-back of their lanes (~3.6 us per symbol: 21 planes of 8-byte pieces) stays small
    // (up to a third of the symbols and four rounds of null-aware CTAs in DIRECT mode, launch_suite: no write-back there)
    if (n_x == 0 || n_xb * 2 > p->n_null_blocks || n_xb > 4 * p->e->sm_count || n_x * 3 > p->n_symbols) return PQB_OK;
    map.resize((size_t)(n_xb * SYM), -1);
    p->h_xstart.assign(map.size(), 0);
    p->h_xflags.assign(map.size(), 0);
    for (size_t i = 0; i < map.size(); ++i)
        if (map[i] >= 0) { p->h_xstart[i] = p->h_start_explicit[(size_t)map[i]]; p->h_xflags[i] = p->h_flags[(size_t)map[i]]; }
    if (n_xb > p->x_cap_blocks) {                       // (re)allocate the compacted planes
        for (auto &q : p->x_in) if (q) { cudaFree(q); q = nullptr; }
        for (auto &q : p->x_out) if (q) { cudaFree(q); q = nullptr; }
        for (auto &q : p->x_ovm) if (q) { cudaFree(q); q = nullptr; }
        if (p->x_vmask) { cudaFree(p->x_vmask); p->x_vmask = nullptr; }
        if (p->d_symmap) { cudaFree(p->d_symmap); p->d_symmap = nullptr; }
        if (p->d_xstart) { cudaFree(p->d_xstart); p->d_xstart = nullptr; }
        if (p->d_xflags) { cudaFree(p->d_xflags); p->d_xflags = nullptr; }
        const int64_t cap = n_xb + n_xb / 4 + 1;
        const size_t xplane = (size_t)cap * p->bars_padded * SYM * sizeof(double), xwords = (size_t)cap * p->bars_padded;
        for (int f = 0; f < PQB_N_FIELDS; ++f) if (p->d_in[f]) CU(cudaMalloc(&p->x_in[f], xplane));
        for (int k = 0; k < PQB_N_OUTPUTS; ++k)
            if (p->d_out[k]) { CU(cudaMalloc(&p->x_out[k], xplane)); CU(cudaMalloc(&p->x_ovm[k], xwords * sizeof(uint32_t))); }
        CU(cudaMalloc(&p->x_vmask, xwords * N_IN * sizeof(uint32_t)));
        CU(cudaMalloc(&p->d_symmap, (size_t)cap * SYM * sizeof(int)));
        CU(cudaMalloc(&p->d_xstart, (size_t)cap * SYM * sizeof(int)));
        CU(cudaMalloc(&p->d_xflags, (size_t)cap * SYM));
        p->x_cap_blocks = cap;
    }
    if (!p->d_start_c) CU(cudaMalloc(&p->d_start_c, (size_t)p->n_blocks * SYM * sizeof(int)));
    CU(cudaMemcpyAsync(p->d_symmap, map.data(), map.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(p->d_xstart, p->h_xstart.data(), map.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(p->d_xflags, p->h_xflags.data(), map.size(), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(p->d_start_c, p->h_start_c.data(), (size_t)p->n_symbols * sizeof(int), cudaMemcpyHostToDevice, st));
    // the compacted blocks' input validity words, from the flagged symbols' own row bitmaps
    MaskArgs V{};
    for (int f = 0; f < PQB_N_FIELDS; ++f) V.rm[f] = p->h_vin[f].empty() ? nullptr : p->d_vin[f];
    V.tiled_out = p->x_vmask;
    V.start = p->d_xstart;
    V.symmap = p->d_symmap;
    V.n_symbols = (int)p->n_symbols; V.n_bars = (int)p->n_bars; V.bars_padded = (int)p->bars_padded;
    V.words_per_row = (int)p->words_per_row; V.n_blocks = (int)n_xb;
    V.block0 = 0; V.blist = nullptr;
    dim3 grid((unsigned)((p->bars_padded + 31) / 32), (unsigned)n_xb);
    pack_mask_kernel<<<grid, 32, 0, st>>>(V);
    CU(cudaGetLastError());
    p->n_x = n_x;
    p->n_xblocks = n_xb;
    p->compact = true;
    return PQB_OK;
}

// Per symbol block of the range [s0, s0 + ns) (s0 a multiple of 32): plain (every symbol valid on [start, n_bars), all
// fields alike -> the plain kernels, leading nulls folded into `start`) or null-aware (some symbol of the block has an
// interior / trailing null, or fields starting at different rows -> per-bar validity words, the null-aware kernel).
// The choice is per BLOCK (launch_suite makes one launch per kind over block lists), derived from what the columns
// currently hold -- nothing sticky: overwriting a column with a null-free one returns its block to the plain kernel.
// Ships starts / masks / flags of the range to the device on stream `st`.
// host half: which blocks need the null-aware kernel, the per-symbol starts; returns whether any block of the range does
static bool prepare_nulls_host(pqb_panel *p, int64_t s0, int64_t ns) {
    const int64_t b0 = s0 / SYM, b1 = (s0 + ns + SYM - 1) / SYM;
    bool any_null = false;
    for (int64_t b = b0; b < b1; ++b) {
        bool nulls = false;
        const size_t lo = (size_t)b * SYM, hi = (size_t)std::min<int64_t>((b + 1) * SYM, p->n_symbols);
        for (size_t s = lo; s < hi && !nulls; ++s) {
            if (p->h_flags[s]) { nulls = true; break; }
            int32_t lead = -2;
            for (int f = 0; f < PQB_N_FIELDS; ++f) {
                if (!p->d_in[f] || p->h_lead[f][s] < 0) continue;
                if (lead == -2) lead = p->h_lead[f][s];
                else if (lead != p->h_lead[f][s]) nulls = true;      // fields of one symbol start at different rows
            }
        }
        p->n_null_blocks += (int64_t)nulls - (int64_t)p->h_blk_null[(size_t)b];
        p->h_blk_null[(size_t)b] = nulls ? 1 : 0;
        any_null |= nulls;
        for (size_t s = lo; s < hi; ++s) {
            int32_t a = p->h_start_explicit[s];
            if (!nulls)
                for (int f = 0; f < PQB_N_FIELDS; ++f)
                    if (p->d_in[f]) a = std::max(a, p->h_lead[f][s]);
            p->h_start[s] = a;
            if (a) p->starts_nonzero = true;                         // (sticky within a panel's life: only costs a pointer)
        }
    }
    p->nulls_mode = p->n_null_blocks > 0;
    p->compact = false;
    return any_null;
}
// device half (copy_start = false: the caller's pack launch writes the starts itself, run_single's mapped path)
static int prepare_nulls_device(pqb_panel *p, cudaStream_t st, int64_t s0, int64_t ns, bool any_null, bool copy_start) {
    const int64_t b0 = s0 / SYM, b1 = (s0 + ns + SYM - 1) / SYM;
    if (copy_start)
        CU(cudaMemcpyAsync(p->d_start + s0, p->h_start.data() + s0, (size_t)ns * sizeof(int), cudaMemcpyHostToDevice, st));
    if (!any_null) return PQB_OK;
    const size_t bplane = (size_t)p->n_symbols * p->words_per_row * sizeof(uint32_t);
    const size_t mwords = (size_t)p->n_blocks * p->bars_padded;
    if (!p->d_vmask) CU(cudaMalloc(&p->d_vmask, mwords * N_IN * sizeof(uint32_t)));
    if (!p->d_flags) { CU(cudaMalloc(&p->d_flags, (size_t)p->n_blocks * SYM)); CU(cudaMemsetAsync(p->d_flags, 0, (size_t)p->n_blocks * SYM, st)); }
    CU(cudaMemcpyAsync(p->d_flags + s0, p->h_flags.data() + s0, (size_t)ns, cudaMemcpyHostToDevice, st));
    MaskArgs V{};
    const size_t roff = (size_t)s0 * p->words_per_row, rbytes = (size_t)ns * p->words_per_row * sizeof(uint32_t);
    for (int f = 0; f < PQB_N_FIELDS; ++f) {
        if (p->h_vin[f].empty()) continue;
        if (!p->d_vin[f]) CU(cudaMalloc(&p->d_vin[f], bplane));
        CU(cudaMemcpyAsync(p->d_vin[f] + roff, p->h_vin[f].data() + roff, rbytes, cudaMemcpyHostToDevice, st));
        V.rm[f] = p->d_vin[f];
    }
    for (int k = 0; k < PQB_N_OUTPUTS; ++k)
        if (p->d_out[k] && !p->d_ovm[k]) CU(cudaMalloc(&p->d_ovm[k], mwords * sizeof(uint32_t)));
    V.tiled_out = p->d_vmask;
    V.start = p->d_start;
    V.n_symbols = (int)p->n_symbols; V.n_bars = (int)p->n_bars; V.bars_padded = (int)p->bars_padded;
    V.words_per_row = (int)p->words_per_row; V.n_blocks = (int)p->n_blocks;
    V.block0 = (int)b0; V.blist = nullptr;
    dim3 grid((unsigned)((p->bars_padded + 31) / 32), (unsigned)(b1 - b0));
    pack_mask_kernel<<<grid, 32, 0, st>>>(V);
    CU(cudaGetLastError());
    if (s0 == 0 && ns == p->n_symbols) return prepare_compaction(p, st);
    return PQB_OK;
}
static int prepare_nulls(pqb_panel *p, cudaStream_t st, int64_t s0 = 0, int64_t ns = -1) {
    if (ns < 0) ns = p->n_symbols - s0;
    return prepare_nulls_device(p, st, s0, ns, prepare_nulls_host(p, s0, ns), true);
}

// ---- layout conversion launches (chunk = symbols [s0, s0+ns), s0 a multiple of 32) ----
static int launch_conv(pqb_panel *p, bool pack, const double *const *rowmajor, double *const *tiled, int n_planes,
                       int64_t s0, int64_t ns, cudaStream_t st, const ConvArgs *extra = nullptr) {
    if (n_planes == 0 || ns == 0) return PQB_OK;
    ConvArgs V{};
    if (extra) V = *extra;                                    // (riders of run_single's mapped path: starts / validity words)
    V.n_planes = n_planes;
    for (int i = 0; i < n_planes; ++i) {
        if (pack) { V.src[i] = rowmajor[i]; V.dst[i] = tiled[i]; }
        else { V.src[i] = tiled[i]; V.dst[i] = const_cast<double *>(rowmajor[i]); }
    }
    V.n_symbols = (int)ns;
    V.n_bars = (int)p->n_bars;
    V.pitch = (int)p->pitch;
    V.bars_padded = (int)p->bars_padded;
    V.block0 = (int)(s0 / SYM);
    dim3 grid((unsigned)((p->bars_padded + 31) / 32), (unsigned)((ns + SYM - 1) / SYM));
    if (pack) pack_kernel<<<grid, 256, 0, st>>>(V);
    else unpack_kernel<<<grid, 256, 0, st>>>(V);
    CU(cudaGetLastError());
    return PQB_OK;
}

extern "C" int pqb_panel_upload(pqb_panel *p) {
    if (!p || !p->staging) return fail(PQB_ERR_INVALID, "pqb_panel_upload: no host staging");
    int rc = set_dev(p->e);
    if (rc) return rc;
    cudaStream_t st = p->e->stream;
    const size_t cplane = (size_t)p->chunk_symbols * p->pitch;
    for (int64_t s0 = 0; s0 < p->n_symbols; s0 += p->chunk_symbols) {
        const int64_t ns = std::min(p->chunk_symbols, p->n_symbols - s0);
        const double *rm[PQB_N_FIELDS];
        double *tl[PQB_N_FIELDS];
        int n = 0;
        for (int f = 0; f < PQB_N_FIELDS; ++f) {
            if (!p->d_in[f]) continue;
            double *buf = p->d_xin[0] + cplane * p->in_slot[f];
            CU(cudaMemcpyAsync(buf, p->h_in[f] + (size_t)s0 * p->pitch, (size_t)ns * p->pitch * sizeof(double),
                               cudaMemcpyHostToDevice, st));
            rm[n] = buf; tl[n] = p->d_in[f]; ++n;
        }
        if ((rc = launch_conv(p, true, rm, tl, n, s0, ns, st))) return rc;
    }
    p->inputs_resident = true;
    return prepare_nulls(p, st);
}

// tiled device planes -> pinned row-major staging (outputs + validity, or the input fields)
static int download_planes(pqb_panel *p, bool inputs) {
    cudaStream_t st = p->e->stream;
    const size_t cplane = (size_t)p->chunk_symbols * p->pitch;
    for (int64_t s0 = 0; s0 < p->n_symbols; s0 += p->chunk_symbols) {
        const int64_t ns = std::min(p->chunk_symbols, p->n_symbols - s0);
        const double *rm[PQB_N_OUTPUTS];
        double *tl[PQB_N_OUTPUTS];
        double *host[PQB_N_OUTPUTS];
        int n = 0;
        if (inputs) {
            for (int f = 0; f < PQB_N_FIELDS; ++f)
                if (p->d_in[f]) { rm[n] = p->d_xin[0] + cplane * p->in_slot[f]; tl[n] = p->d_in[f]; host[n] = p->h_in[f]; ++n; }
        } else {
            for (int k = 0; k < PQB_N_OUTPUTS; ++k)
                if (p->d_out[k]) { rm[n] = p->d_xout[0] + cplane * p->out_slot[k]; tl[n] = p->d_out[k]; host[n] = p->h_out[k]; ++n; }
        }
        int rc = launch_conv(p, false, rm, tl, n, s0, ns, st);
        if (rc) return rc;
        for (int i = 0; i < n; ++i)
            CU(cudaMemcpyAsync(host[i] + (size_t)s0 * p->pitch, rm[i], (size_t)ns * p->pitch * sizeof(double),
                               cudaMemcpyDeviceToHost, st));
    }
    if (!inputs) {
        const size_t bplane = (size_t)p->n_symbols * p->words_per_row * sizeof(uint32_t);
        for (int k = 0; k < PQB_N_OUTPUTS; ++k)
            if (p->d_out[k]) CU(cudaMemcpyAsync(p->h_bits[k], p->d_bits[k], bplane, cudaMemcpyDeviceToHost, st));
    }
    return PQB_OK;
}

extern "C" int pqb_panel_download(pqb_panel *p) {
    if (!p || !p->staging) return fail(PQB_ERR_INVALID, "pqb_panel_download: no host staging");
    int rc = set_dev(p->e);
    if (rc) return rc;
    return download_planes(p, false);
}

extern "C" int pqb_panel_sync(pqb_panel *p) {
    if (!p) return fail(PQB_ERR_INVALID, "pqb_panel_sync: NULL");
    int rc = set_dev(p->e);
    if (rc) return rc;
    CU(cudaStreamSynchronize(p->e->h2d));
    CU(cudaStreamSynchronize(p->e->stream));
    CU(cudaStreamSynchronize(p->e->d2h));
    return PQB_OK;
}

extern "C" int pqb_panel_get_output(pqb_panel *p, int64_t symbol, int output, double *values, uint8_t *validity,
                                    int64_t len) {
    if (!p || !values) return fail(PQB_ERR_INVALID, "pqb_panel_get_output: NULL argument");
    if (!p->staging || output < 0 || output >= PQB_N_OUTPUTS || !p->h_out[output] || symbol < 0 ||
        symbol >= p->n_symbols || len != p->n_bars)
        return fail(PQB_ERR_INVALID, "pqb_panel_get_output: bad symbol/output/len");
    memcpy(values, p->h_out[output] + (size_t)symbol * p->pitch, (size_t)len * sizeof(double));
    if (validity)
        memcpy(validity, reinterpret_cast<const uint8_t *>(p->h_bits[output] + (size_t)symbol * p->words_per_row),
               (size_t)((len + 7) / 8));
    return PQB_OK;
}

// ---------------------------------------------------------------------------------------
// parameters -> kernel arguments
// ---------------------------------------------------------------------------------------
static inline double ema_alpha(int p) { return 2.0 / ((double)p + 1.0); }   // overlap.rs:669

struct Built {
    SuiteArgs a;
    int lead[PQB_N_OUTPUTS];   // first valid index of each output relative to the symbol start
    int steady_b;              // a.steady_lead of the benchmark groups alone (their own null-aware launch next to optional groups)
};

static bool split_launch_enabled() {
    const char *s = getenv("PQB_SPLIT_LAUNCH");           // (0: one general launch for everything -- measurement knob)
    return !s || atoi(s) != 0;
}

// panels of up to this many symbol blocks run the small-panel variant of the full suite (nine pipelined role warps, two
// CTAs per SM); PQB_SMALL_BLOCKS overrides (tuning)
// CTAs per tail block: as many as keeps the tail launch at about half a CTA per SM (measured, profiles/r03a_compact_tail.txt:
// 9 tail blocks -> one role per CTA, 24 -> three roles per CTA; more tail CTAs than that cost more than they spread)
static int tail_parts_compact(const pqb_engine *e, int64_t n_tail) {
    static const int forced = getenv("PQB_TAIL_PARTS") ? std::max(1, std::min((int)N_ROLES_X, atoi(getenv("PQB_TAIL_PARTS")))) : 0;
    if (forced) return forced;
    const int64_t by_budget = (e->sm_count * 55ll / 100) / std::max<int64_t>(n_tail, 1);
    return (int)std::max<int64_t>(2, std::min<int64_t>(N_ROLES_X, by_budget));
}
static bool tail_compact() {
    static const bool v = !getenv("PQB_TAIL_COMPACT") || atoi(getenv("PQB_TAIL_COMPACT")) != 0;
    return v;
}
static int64_t small_max_blocks(const pqb_engine *e) {
    static const char *ev = getenv("PQB_SMALL_BLOCKS");
    if (ev) return atoll(ev);
    // one whole-block CTA per SM + up to sm_count / 5 blocks beyond as compact tail CTAs (beyond that the plain kernel with two
    // CTAs on some SMs is as fast: 196 blocks 1.61 against 1.59 ms)
    if (tail_compact()) return e->sm_count + e->sm_count / 5;
    return e->sm_count + e->sm_count / N_ROLES_X;
}

// shared-memory ring layout of one launch: offsets of every enabled group's rings / van Herk arrays and the dynamic
// shared-memory size (depends on A.gmask and the periods only, so a launch of a subset of the groups gets its own)
static int layout_rings(SuiteArgs &A, const pqb_panel *p) {
    // shared-memory rings (slots of 32 doubles)
    const bool mid_shares = (A.gmask & G_WILLR) && A.willr_p == A.mid_p;
    // MIDPRICE shares WILLR's arrays when the windows are equal -- except for the full suite on a small panel, where the
    // nine-warp variant runs it in a warp of its own (launch_suite picks that variant only if these arrays exist)
    // ... and for a partial suite in the latency regime (at most one wave of three CTAs per SM) with a role warp to spare,
    // where deal_base_slots() gives WILLR and MIDPRICE a warp each
    int active_roles = 0;
    for (int r = 0; r < N_ROLES; ++r) active_roles += (A.gmask & ROLE_GROUPS[r]) ? 1 : 0;
    const bool partial_spare = !(A.gmask & ~(unsigned)G_ALL) && A.gmask != (unsigned)G_ALL && active_roles < N_ROLES &&
                               p->n_blocks <= 3ll * p->e->sm_count;
    A.mid_own = (A.gmask & G_MIDPRICE) &&
                (!mid_shares || partial_spare || (A.gmask == G_ALL && p->n_blocks <= small_max_blocks(p->e)));
retry_layout:
    long long off = 0;
    auto take = [&](int slots) { const long long o = off; off += (long long)std::max(slots, 1) * SYM; return (int)std::min<long long>(o, 1ll << 30); };
    A.sring_slots = (A.gmask & G_SMA) ? A.sma_p : 1; A.off_sring = take(A.sring_slots);
    A.bring_slots = (A.gmask & G_BB) ? A.bb_p : 1; A.off_bring = take(A.bring_slots);
    A.c1ring_slots = (A.gmask & G_TRIMA) ? A.tri_n1 : 1; A.off_c1ring = take(A.c1ring_slots);
    A.tring_slots = (A.gmask & G_TRIMA) ? A.tri_n2 : 1; A.off_tring = take(A.tring_slots);
    A.fk_slots = (A.gmask & G_KDJ) ? A.kdj_sk : 1; A.off_fk = take(A.fk_slots);
    A.sk_slots = (A.gmask & G_KDJ) ? A.kdj_sd : 1; A.off_sk = take(A.sk_slots);
    // van Herk arrays: p slots + 1 sentinel each
    const int wp = (A.gmask & G_WILLR) ? A.willr_p + 1 : 0;
    const int mp = A.mid_own ? A.mid_p + 1 : 0;
    const int kp = (A.gmask & G_KDJ) ? A.kdj_k + 1 : 0;
    A.off_wh = take(wp); A.off_wl = take(wp);
    A.off_mh = take(mp); A.off_ml = take(mp);
    A.off_kh = take(kp); A.off_kl = take(kp);
    A.off_mom = take((A.gmask & G_MOM) ? A.mom_p : 0);
    A.off_roc = take((A.gmask & G_ROC) ? A.roc_p : 0);
    A.off_cmou = take((A.gmask & G_CMO) ? A.cmo_p : 0); A.off_cmod = take((A.gmask & G_CMO) ? A.cmo_p : 0);
    A.off_mfip = take((A.gmask & G_MFI) ? A.mfi_p : 0); A.off_mfin = take((A.gmask & G_MFI) ? A.mfi_p : 0);
    A.off_cci = take((A.gmask & G_CCI) ? A.cci_p : 0);
    A.off_mph = take((A.gmask & G_MIDPOINT) ? A.midpoint_p + 1 : 0); A.off_mpl = take((A.gmask & G_MIDPOINT) ? A.midpoint_p + 1 : 0);
    A.off_adx = take((A.gmask & G_DM) ? A.dm_p - 1 : 0);
    A.off_ult = take((A.gmask & G_ULTOSC) ? 2 * std::max(std::max(A.ult_p1, A.ult_p2), A.ult_p3) : 2);
    A.off_arh = take((A.gmask & G_AROON) ? A.aroon_p + 1 : 0); A.off_arl = take((A.gmask & G_AROON) ? A.aroon_p + 1 : 0);
    A.off_ari = take((A.gmask & G_AROON) ? (A.aroon_p + 2) / 2 : 0);      // packed offsets of the suffix extremes: 4 bytes per lane and slot
    A.off_art = take((A.gmask & G_AROON) ? (A.aroon_p + SYM) / SYM : 0);    // the p + 1 quotients (position / p) * 100
    A.off_dh = take((A.gmask & G_DONCHIAN) ? A.don_p + 1 : 0); A.off_dl = take((A.gmask & G_DONCHIAN) ? A.don_p + 1 : 0);
    const long long smem = (long long)kFixedSmem + off * 8;
    if (smem > kMaxSmem && A.mid_own && mid_shares) { A.mid_own = 0; goto retry_layout; }   // long windows: share after all
    if (smem > kSmemThreeCtas && A.mid_own && mid_shares && partial_spare) { A.mid_own = 0; goto retry_layout; }   // (not at the cost of a CTA per SM)
    if (smem > kMaxSmem)
        return fail(PQB_ERR_UNSUPPORTED,
                    "windows too long for one launch: the per-block rings need %lld bytes of shared memory (limit %d); "
                    "run long-window indicators in separate calls", smem, kMaxSmem);
    A.smem_bytes = (int)smem;
    return PQB_OK;
}

// roles with work and input planes to stage, from the enabled groups
static void derive_roles(SuiteArgs &A) {
    A.roles = 0; A.n_roles = 0; A.fields = 0;
    for (int r = 0; r < N_ROLES; ++r)
        if (A.gmask & ROLE_GROUPS[r]) { A.roles |= 1u << r; ++A.n_roles; }
    if (A.gmask & ~(unsigned)(G_MIDPRICE | G_DONCHIAN)) A.fields |= F_C;        // everything but midprice / donchian reads close
    if (A.gmask & (G_TRANGE | G_ATR | G_NATR | G_AD | G_KDJ | G_WILLR | G_MIDPRICE | G_ADOSC | G_MFI | G_CCI | G_DM | G_ULTOSC | G_AROON | G_DONCHIAN)) A.fields |= F_H | F_L;
    if (A.gmask & (G_OBV | G_AD | G_ADOSC | G_MFI)) A.fields |= F_V;
}

static int build_args(const pqb_panel *p, const pqb_suite_params *sp, Built *out) {
    SuiteArgs &A = out->a;
    memset(out, 0, sizeof *out);
    const int n_bars = (int)p->n_bars;
    const int NEVER = n_bars;                       // lead that makes a column all-null
    uint32_t ind = sp->indicators & (PQB_IND_ALL | PQB_IND_EXTRAS);
    auto need_fields = [&](uint32_t mask, const char *what) -> int {
        if ((p->fields_mask & mask) != mask) return fail(PQB_ERR_INVALID, "%s needs panel fields 0x%x", what, mask);
        return PQB_OK;
    };
    const uint32_t C = 1u << PQB_CLOSE, H = 1u << PQB_HIGH, L = 1u << PQB_LOW, V = 1u << PQB_VOLUME;
    int rc;
    if ((ind & (PQB_IND_SMA | PQB_IND_EMA | PQB_IND_TEMA | PQB_IND_TRIMA | PQB_IND_BBANDS | PQB_IND_MACD | PQB_IND_RSI)) &&
        (rc = need_fields(C, "close-based indicators"))) return rc;
    if ((ind & (PQB_IND_TRANGE | PQB_IND_ATR | PQB_IND_NATR | PQB_IND_KDJ | PQB_IND_WILLR)) &&
        (rc = need_fields(C | H | L, "high/low/close indicators"))) return rc;
    if ((ind & PQB_IND_MIDPRICE) && (rc = need_fields(H | L, "midprice"))) return rc;
    if ((ind & PQB_IND_OBV) && (rc = need_fields(C | V, "obv"))) return rc;
    if ((ind & (PQB_IND_AD | PQB_IND_ADOSC | PQB_IND_MFI)) && (rc = need_fields(C | H | L | V, "ad / adosc / mfi"))) return rc;
    if ((ind & (PQB_IND_MIDPOINT | PQB_IND_MOM | PQB_IND_ROC | PQB_IND_CMO)) && (rc = need_fields(C, "close-based indicators"))) return rc;
    if ((ind & PQB_IND_CCI) && (rc = need_fields(C | H | L, "cci"))) return rc;

    for (int f = 0; f < PQB_N_FIELDS; ++f) A.in[f] = p->d_in[f];
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) { A.out[k] = nullptr; out->lead[k] = NEVER; }
    A.don_fold = 0; A.don_p = 1;
    // the arguments of the PLAIN kernels; launch_suite derives the null-aware variant (null_variant) for the symbol
    // blocks that need it
    A.symmap = nullptr;
    A.start = p->d_start;      // (always: with pipelined intake the starts reach the device after these arguments are built)
    A.vmask = nullptr;
    A.symflags = nullptr;
    A.blist = nullptr;
    // validity words: the optional groups always (roc / cci decide per bar); every output in the null-aware variant
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) A.ovm[k] = (k >= PQB_N_SUITE_OUTPUTS) ? p->d_ovm[k] : nullptr;
    A.n_symbols = (int)p->n_symbols;
    A.n_bars = n_bars;
    A.n_blocks = (int)p->n_blocks;
    A.bars_padded = (int)p->bars_padded;
    A.block0 = 0;

    int steady = 1;
    auto neg = [&](int v, const char *name) -> int {
        return v < 0 ? fail(PQB_ERR_INVALID, "%s period %d is negative", name, v) : PQB_OK;
    };
    auto want = [&](int k) { return p->d_out[k] != nullptr; };
    auto bind = [&](int k, long long lead) {
        if (want(k)) { A.out[k] = p->d_out[k]; out->lead[k] = (int)std::min<long long>(lead, NEVER); }
    };
    // A period of 0 makes the reference return an all-null column (guards overlap.rs:663,874,...):
    // the output is bound with lead = NEVER and its group stays off (run_suite NaN-fills it).
    auto null_only = [&](int k) { if (want(k)) { A.out[k] = p->d_out[k]; out->lead[k] = NEVER; } };
    auto upto = [&](long long j) { steady = (int)std::min<long long>(std::max<long long>(steady, j), 1ll << 30); };

    if (ind & PQB_IND_SMA) {
        if ((rc = neg(sp->sma_period, "sma"))) return rc;
        if (sp->sma_period == 0) { null_only(PQB_OUT_SMA); }
        else { A.gmask |= G_SMA; A.sma_p = sp->sma_period; A.inv_sma = 1.0 / (double)sp->sma_period;
               bind(PQB_OUT_SMA, sp->sma_period - 1); upto(sp->sma_period); }
    }
    if (ind & PQB_IND_TEMA) {
        if ((rc = neg(sp->tema_period, "tema"))) return rc;
        const int tp = sp->tema_period;
        // guard overlap.rs:1180: n < 3p-2 -> all null (equivalent to lead >= n)
        if (tp == 0) { null_only(PQB_OUT_TEMA); }
        // tp == 1: the reference's `count == p` branch wins over `count == 3p-2` -> first value at index 1
        else { A.gmask |= G_TEMA; A.tema_p = tp; A.a_tema = ema_alpha(tp);
               bind(PQB_OUT_TEMA, tp == 1 ? 1 : 3ll * tp - 3); upto(tp == 1 ? 2 : 3ll * tp - 2); }
    }
    if (ind & PQB_IND_EMA) {
        if ((rc = neg(sp->ema_period, "ema"))) return rc;
        const int ep = sp->ema_period;
        if (ep == 0) { null_only(PQB_OUT_EMA); }
        else { A.gmask |= G_EMA; A.ema_p = ep; A.a_ema = ema_alpha(ep); bind(PQB_OUT_EMA, ep - 1); upto(ep); }
    }
    if (ind & PQB_IND_TRIMA) {
        if ((rc = neg(sp->trima_period, "trima"))) return rc;
        const int tp = sp->trima_period;
        int n1, n2;
        if (tp % 2 == 1) { n1 = tp / 2 + 1; n2 = n1; } else { n1 = tp / 2; n2 = n1 + 1; }   // overlap.rs:1314-1323
        if (n1 == 0) { null_only(PQB_OUT_TRIMA); }
        else { A.gmask |= G_TRIMA; A.tri_n1 = n1; A.tri_n2 = n2; A.inv_tri1 = 1.0 / (double)n1; A.inv_tri2 = 1.0 / (double)n2;
               bind(PQB_OUT_TRIMA, (long long)n1 + n2 - 2); upto((long long)n1 + n2 - 1); }
    }
    if (ind & PQB_IND_BBANDS) {
        if ((rc = neg(sp->bbands_period, "bbands"))) return rc;
        const int bp = sp->bbands_period;
        if (bp == 0) { for (int k = 4; k <= 6; ++k) { null_only(k); } }
        else { A.gmask |= G_BB; A.bb_p = bp; A.bb_pd = (double)bp;
               A.bb_up = sp->bbands_nbdevup; A.bb_dn = sp->bbands_nbdevdn;
               for (int k = 4; k <= 6; ++k) bind(k, bp - 1);
               upto(bp); }
    }
    if (ind & PQB_IND_MACD) {
        const int f = sp->macd_fast, s = sp->macd_slow, g = sp->macd_signal;
        if ((rc = neg(f, "macd fast")) || (rc = neg(s, "macd slow")) || (rc = neg(g, "macd signal"))) return rc;
        if (f == 0 || s == 0 || g == 0)
            return fail(PQB_ERR_UNSUPPORTED, "macd with a zero period (reference yields partial nulls) is not built");
        A.gmask |= G_MACD;
        A.macd_f = f; A.macd_s = s; A.macd_g = g;
        A.a_mf = ema_alpha(f); A.a_ms = ema_alpha(s); A.a_mg = ema_alpha(g);
        const int dl = std::max(f, s) - 1;
        bind(PQB_OUT_MACD, dl); bind(PQB_OUT_MACD_SIGNAL, g - 1);
        bind(PQB_OUT_MACD_HIST, std::max(dl, g - 1));
        upto(std::max(std::max(f, s), g));
    }
    if (ind & PQB_IND_RSI) {
        if ((rc = neg(sp->rsi_period, "rsi"))) return rc;
        const int rp = sp->rsi_period;
        if (rp == 0) { null_only(PQB_OUT_RSI); }
        else { A.gmask |= G_RSI; A.rsi_p = rp; A.a_rsi = 1.0 / (double)rp; bind(PQB_OUT_RSI, rp - 1); upto(rp); }   // D1
    }
    if (ind & PQB_IND_TRANGE) { A.gmask |= G_TRANGE; bind(PQB_OUT_TRANGE, 1); }
    if (ind & PQB_IND_ATR) {
        if (sp->atr_period <= 0) return fail(PQB_ERR_INVALID, "atr period %d: 2p-1 underflows in the reference", sp->atr_period);
        const int ep = 2 * sp->atr_period - 1;                                               // volatility.rs:30
        A.gmask |= G_ATR; A.atr_ep = ep; A.a_atr = ema_alpha(ep); bind(PQB_OUT_ATR, (long long)ep); upto((long long)ep + 1);
    }
    if (ind & PQB_IND_NATR) {
        if (sp->natr_period <= 0) return fail(PQB_ERR_INVALID, "natr period %d: 2p-1 underflows in the reference", sp->natr_period);
        const int ep = 2 * sp->natr_period - 1;
        A.gmask |= G_NATR; A.natr_ep = ep; A.a_natr = ema_alpha(ep); bind(PQB_OUT_NATR, (long long)ep); upto((long long)ep + 1);
    }
    if (ind & PQB_IND_OBV) { A.gmask |= G_OBV; bind(PQB_OUT_OBV, 1); }
    if (ind & PQB_IND_AD) { A.gmask |= G_AD; bind(PQB_OUT_AD, 0); }
    if (ind & PQB_IND_KDJ) {
        const int k = sp->kdj_fastk, sk = sp->kdj_slowk, sd = sp->kdj_slowd;
        if ((rc = neg(k, "kdj fastk")) || (rc = neg(sk, "kdj slowk")) || (rc = neg(sd, "kdj slowd"))) return rc;
        if (k == 0 || sk == 0 || sd == 0) {
            for (int q = 16; q <= 18; ++q) { null_only(q); }
            if (k != 0 && sk != 0 && sd == 0)
                return fail(PQB_ERR_UNSUPPORTED, "kdj with slowd_period 0 (K valid, D null) is not built");
        } else {
            A.gmask |= G_KDJ; A.kdj_k = k; A.kdj_sk = sk; A.kdj_sd = sd; A.inv_sk = 1.0 / (double)sk; A.inv_sd = 1.0 / (double)sd;
            bind(PQB_OUT_KDJ_K, (long long)k + sk - 2); bind(PQB_OUT_KDJ_D, (long long)k + sk + sd - 3);
            bind(PQB_OUT_KDJ_J, (long long)k + sk + sd - 3);
            if ((sp->indicators & PQB_IND_FASTK) && want(PQB_OUT_FASTK)) { A.out[PQB_OUT_FASTK] = p->d_out[PQB_OUT_FASTK]; out->lead[PQB_OUT_FASTK] = NEVER; }   // validity from the kernel
            upto((long long)k + sk + sd - 2);
        }
    }
    if (ind & PQB_IND_WILLR) {
        if ((rc = neg(sp->willr_period, "willr"))) return rc;
        if (sp->willr_period == 0) { null_only(PQB_OUT_WILLR); }
        else { A.gmask |= G_WILLR; A.willr_p = sp->willr_period; bind(PQB_OUT_WILLR, sp->willr_period - 1); upto(sp->willr_period); }
    }
    if (ind & PQB_IND_MIDPRICE) {
        if (sp->midprice_period <= 0)
            return fail(PQB_ERR_UNSUPPORTED, "midprice period %d (reference: never-expiring deque) is not built", sp->midprice_period);
        A.gmask |= G_MIDPRICE; A.mid_p = sp->midprice_period; bind(PQB_OUT_MIDPRICE, 0);
    }
    out->steady_b = steady;
    // ---- optional groups (SURVEY.md 8a, not part of the benchmark suite) ----
    auto bind_dyn = [&](int k) { if (want(k)) { A.out[k] = p->d_out[k]; out->lead[k] = NEVER; } };   // validity from the kernel
    if (ind & PQB_IND_MIDPOINT) {
        if (sp->midpoint_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "midpoint period %d (reference: never-expiring deque) is not built", sp->midpoint_period);
        A.gmask |= G_MIDPOINT; A.midpoint_p = sp->midpoint_period; bind_dyn(PQB_OUT_MIDPOINT);
    }
    if (ind & PQB_IND_ADOSC) {
        const int f = sp->adosc_fast, sl = sp->adosc_slow;
        if (f <= 0 || sl <= 0) return fail(PQB_ERR_UNSUPPORTED, "adosc with a period <= 0 is not built");
        A.gmask |= G_ADOSC; A.adosc_f = f; A.adosc_s = sl; A.a_adf = ema_alpha(f); A.a_ads = ema_alpha(sl);
        bind_dyn(PQB_OUT_ADOSC); upto(std::max(f, sl));
    }
    if (ind & PQB_IND_MOM) {
        if (sp->mom_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "mom period %d <= 0 is not built", sp->mom_period);
        A.gmask |= G_MOM; A.mom_p = sp->mom_period; bind_dyn(PQB_OUT_MOM); upto(sp->mom_period);
    }
    if (ind & PQB_IND_ROC) {
        if (sp->roc_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "roc period %d <= 0 is not built", sp->roc_period);
        A.gmask |= G_ROC; A.roc_p = sp->roc_period; upto(sp->roc_period);
        for (int k = PQB_OUT_ROC; k <= PQB_OUT_ROCR100; ++k) bind_dyn(k);
    }
    if (ind & PQB_IND_CMO) {
        if (sp->cmo_period <= 0) { null_only(PQB_OUT_CMO); }                 // momentum.rs: nothing emitted
        else { A.gmask |= G_CMO; A.cmo_p = sp->cmo_period; bind_dyn(PQB_OUT_CMO); upto(sp->cmo_period); }
    }
    if (ind & PQB_IND_MFI) {
        if (sp->mfi_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "mfi period %d <= 0 is not built", sp->mfi_period);
        A.gmask |= G_MFI; A.mfi_p = sp->mfi_period; bind_dyn(PQB_OUT_MFI); upto((long long)sp->mfi_period + 1);
    }
    if (ind & PQB_IND_CCI) {
        if (sp->cci_period <= 0) { null_only(PQB_OUT_CCI); }                 // calc_sma guard: all null
        else { A.gmask |= G_CCI; A.cci_p = sp->cci_period; A.cci_pd = (double)sp->cci_period; A.inv_cci = 1.0 / (double)sp->cci_period;
               bind_dyn(PQB_OUT_CCI); upto(sp->cci_period); }
    }
    if (ind & PQB_IND_DM) {
        if (sp->dm_period <= 0) { for (int k = PQB_OUT_PLUS_DM; k <= PQB_OUT_ADXR; ++k) null_only(k); }   // calc_rma guard (D1)
        else { A.gmask |= G_DM; A.dm_p = sp->dm_period; A.a_dm = 1.0 / (double)sp->dm_period;              // D1: alpha = 1/p
               for (int k = PQB_OUT_PLUS_DM; k <= PQB_OUT_ADXR; ++k) bind_dyn(k);
               upto(2ll * sp->dm_period); }
    }
    if (ind & PQB_IND_TRIX) {
        if (sp->trix_period <= 0) { null_only(PQB_OUT_TRIX); }                                            // calc_ema guard
        else { A.gmask |= G_TRIX; A.trix_p = sp->trix_period; A.a_trix = ema_alpha(sp->trix_period);
               bind_dyn(PQB_OUT_TRIX); upto((long long)sp->trix_period + 1); }
    }
    if (ind & PQB_IND_ULTOSC) {
        if (sp->ultosc_period1 <= 0 || sp->ultosc_period2 <= 0 || sp->ultosc_period3 <= 0)
            return fail(PQB_ERR_UNSUPPORTED, "ultosc with a period <= 0 (usize underflow in the reference) is not built");
        A.gmask |= G_ULTOSC; A.ult_p1 = sp->ultosc_period1; A.ult_p2 = sp->ultosc_period2; A.ult_p3 = sp->ultosc_period3;
        bind_dyn(PQB_OUT_ULTOSC); upto((long long)std::max(std::max(A.ult_p1, A.ult_p2), A.ult_p3) + 1);
    }
    if (ind & PQB_IND_AROON) {
        if (sp->aroon_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "aroon period %d <= 0 (0 / 0 in the reference) is not built", sp->aroon_period);
        A.gmask |= G_AROON; A.aroon_p = sp->aroon_period; A.aroon_pd = (double)sp->aroon_period;
        bind_dyn(PQB_OUT_AROON_UP); bind_dyn(PQB_OUT_AROON_DOWN); upto((long long)sp->aroon_period + 1);
    }
    if (ind & PQB_IND_DONCHIAN) {
        if (sp->donchian_period <= 0) return fail(PQB_ERR_UNSUPPORTED, "donchian period %d <= 0 (a never-expiring window) is not built", sp->donchian_period);
        // next to a MIDPRICE of the same period in a partial suite the two lines are by-products of its window extremes
        // (one launch, no second pass over high / low); otherwise a group of its own in the optional launch
        A.don_p = sp->donchian_period;
        if ((A.gmask & G_MIDPRICE) && A.mid_p == A.don_p && (A.gmask & (unsigned)G_ALL) != (unsigned)G_ALL) A.don_fold = 1;
        else A.gmask |= G_DONCHIAN;
        bind_dyn(PQB_OUT_DONCHIAN_UPPER); bind_dyn(PQB_OUT_DONCHIAN_LOWER);
    }
    for (int k = PQB_N_SUITE_OUTPUTS; k < PQB_N_OUTPUTS; ++k)
        if (A.out[k] && !p->d_ovm[k]) return fail(PQB_ERR_INVALID, "internal: validity words of output %d are not allocated", k);
    A.steady_lead = steady;

    // roles with work, planes to stage
    derive_roles(A);

    // benchmark groups next to optional groups run as two launches, each with its own layout (launch_suite): what has to
    // fit is each half, not their union (e.g. WILLR(250) + MIDPRICE(250) next to DONCHIAN(250))
    const unsigned gb = A.gmask & (unsigned)G_ALL, go = A.gmask & ~(unsigned)G_ALL;
    if (gb && go && !A.vmask && split_launch_enabled()) {
        for (unsigned part : {gb, go}) {
            SuiteArgs t = A;
            t.gmask = part;
            if ((rc = layout_rings(t, p))) return rc;
        }
        A.smem_bytes = 0;                                   // (launch_suite lays each half out again)
        return PQB_OK;
    }
    return layout_rings(A, p);
}

#if defined(PQB_DEBUG_CLOCKS) || defined(PQB_DEBUG_SMID)
static unsigned long long *g_dbg = nullptr;
#endif

// NaN fill for all-null columns (period 0)
__global__ void nan_fill_kernel(double *p, size_t n) {
    const double nn = __longlong_as_double(0x7ff8000000000000LL);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = nn;
}

// which outputs does an enabled group actually store?  (used for the period-0 NaN fill)
static uint64_t outputs_of_groups(unsigned g) {
    uint64_t m = 0;
    if (g & G_SMA) m |= 1u << 0;
    if (g & G_EMA) m |= 1u << 1;
    if (g & G_TEMA) m |= 1u << 2;
    if (g & G_TRIMA) m |= 1u << 3;
    if (g & G_BB) m |= 7u << 4;
    if (g & G_MACD) m |= 7u << 7;
    if (g & G_RSI) m |= 1u << 10;
    if (g & G_TRANGE) m |= 1u << 11;
    if (g & G_ATR) m |= 1u << 12;
    if (g & G_NATR) m |= 1u << 13;
    if (g & G_OBV) m |= 1u << 14;
    if (g & G_AD) m |= 1u << 15;
    if (g & G_KDJ) m |= (7u << 16) | (1ull << 43);        // (fastk: stored by the general and null-aware kernels when bound)
    if (g & G_WILLR) m |= 1u << 19;
    if (g & G_MIDPRICE) m |= 1u << 20;
    if (g & G_MIDPOINT) m |= 1u << 21;
    if (g & G_ADOSC) m |= 1u << 22;
    if (g & G_MOM) m |= 1u << 23;
    if (g & G_ROC) m |= 0xfu << 24;
    if (g & G_CMO) m |= 1u << 28;
    if (g & G_MFI) m |= 1u << 29;
    if (g & G_CCI) m |= 1u << 30;
    if (g & G_DM) m |= 0x3full << 31;
    if (g & G_TRIX) m |= 1ull << 37;
    if (g & G_ULTOSC) m |= 1ull << 38;
    if (g & G_AROON) m |= 3ull << 39;
    if (g & G_DONCHIAN) m |= 3ull << 41;
    return m;
}

// Partial suites: deal the seven role warps of the BASE kernel as (role, groups) slots.  Every active role gets a warp;
// spare warps take one half of a two-part role -- WILLR | MIDPRICE (needs MIDPRICE's own arrays), OBV + TRIMA | AD,
// EMA + TEMA | MACD + SMA, TRANGE + ATR | NATR -- so that a launch with few roles has shorter per-bar chains
// (BASELINE config 5: WILLR + MIDPRICE in two warps instead of one).  A.roles / A.n_roles become the slots with work.
static void deal_base_slots(SuiteArgs &A) {
    static const int order[N_ROLES] = {1, 2, 0, 5, 3, 6, 4};             // warp order of the seven-role kernels
    int n = 0;
    for (int w = 0; w < N_ROLES; ++w) { A.slot_role[w] = 0; A.slot_mask[w] = 0; }
    for (int i = 0; i < N_ROLES; ++i) {
        const unsigned m = A.gmask & ROLE_GROUPS[order[i]];
        if (m) { A.slot_role[n] = order[i]; A.slot_mask[n] = m; ++n; }
    }
    struct Cut { int role; unsigned half; };
    const Cut cuts[] = {{6, (unsigned)(G_MIDPRICE)}, {4, (unsigned)G_AD}, {0, (unsigned)(G_MACD | G_SMA)}, {3, (unsigned)G_NATR}};
    const char *ds = getenv("PQB_DEAL_SLOTS");
    if (!ds || atoi(ds) != 0)
        for (const Cut &c : cuts) {
            if (n >= N_ROLES) break;
            if (c.role == 6 && !A.mid_own) continue;
            for (int w = 0; w < n; ++w) {
                if (A.slot_role[w] != c.role) continue;
                const unsigned a = A.slot_mask[w] & c.half, b = A.slot_mask[w] & ~c.half;
                if (a && b) { A.slot_mask[w] = b; A.slot_role[n] = c.role; A.slot_mask[n] = a; ++n; }
                break;
            }
        }
    // role -> slot code: 3 * role, + 1 for the half without the cut groups, + 2 for the cut half
    for (int w = 0; w < n; ++w) {
        const int role = A.slot_role[w];
        const unsigned whole = A.gmask & ROLE_GROUPS[role];
        int part = 0;
        if (A.slot_mask[w] != whole)
            for (const Cut &c : cuts)
                if (c.role == role) part = (A.slot_mask[w] & c.half) ? 2 : 1;
        A.slot_role[w] = 3 * role + part;
    }
    A.roles = (1u << n) - 1;
    A.n_roles = n;
}

// the null-aware variant of a launch's arguments: per-bar validity words in, per-bar validity words out, starts folded
// into the masks
// fully valid stages of a null-aware launch run the plain steady step (suite_kernel.cuh run_role): only for launches of the 21 suite
// outputs -- the optional outputs report validity per bar through emitv, with null rules of their own (PQB_NULLS_FAST=0: never)
static int nulls_fast_ok(const SuiteArgs &a) {
    static const bool on = !getenv("PQB_NULLS_FAST") || atoi(getenv("PQB_NULLS_FAST")) != 0;
    if (!on || (a.gmask & ~(unsigned)G_ALL) || a.don_fold) return 0;
    for (int k = PQB_N_SUITE_OUTPUTS; k < PQB_N_OUTPUTS; ++k) if (a.out[k]) return 0;
    return 1;
}
static bool nulls_fulls() {              // PQB_NULLS_FULLS=0: the general null-aware kernel also for the full suite
    static const bool on = !getenv("PQB_NULLS_FULLS") || atoi(getenv("PQB_NULLS_FULLS")) != 0;
    return on;
}
static SuiteArgs null_variant(const pqb_panel *p, SuiteArgs a) {
    a.nulls_fast = nulls_fast_ok(a);
    a.start = nullptr;
    a.vmask = p->d_vmask;
    a.symflags = p->d_flags;
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) a.ovm[k] = p->d_ovm[k];
    return a;
}

// tuning: PQB_FULLS_SMEM = dynamic shared memory requested for the full-suite kernel (more than it needs = fewer CTAs per SM)
static int fulls_smem(int need) {
    static const char *ev = getenv("PQB_FULLS_SMEM");
    return ev ? std::max(need, atoi(ev)) : need;
}

// One thread that sleeps ~`ns` nanoseconds on the main stream (PQB_COMPACT_DELAY_US, default 40): the null-aware CTAs of a symbol
// compaction are then resident -- one per SM, each asking for the SM's whole shared memory so that no plain CTA moves in beside
// it -- before the plain grid fills the rest of the GPU.  Measured with a timeline build (globaltimer stamps, profiles/
// r03_halted_symbols.txt): without it they only start when the first plain wave ends (2.0 ms in); sharing an SM with a plain CTA
// their 4.2 ms walk takes 6 - 10 ms (50,000 x 5,040: last null-aware CTA done at 11.7 - 13.4 ms, after the plain launch).
__global__ void delay_kernel(unsigned ns) {
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    do {
        __nanosleep(1000);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    } while (t - t0 < ns);
}

static bool force_base() {
    static const bool v = getenv("PQB_FORCE_BASE") && atoi(getenv("PQB_FORCE_BASE")) != 0;
    return v;
}

// Launches the suite over symbol blocks [b0, b0+nb) (+ NaN fills + validity bitmaps of those symbols).
static int launch_suite(pqb_panel *p, const Built &full, int64_t b0, int64_t nb, cudaEvent_t ev_after_fused,
                        int *launches) {
    pqb_engine *e = p->e;
    int n_launch = 0;
    bool did_compact = false;
    const uint64_t stored = outputs_of_groups(full.a.gmask) | (full.a.don_fold ? 3ull << 41 : 0);
    const size_t boff = (size_t)b0 * p->bars_padded * SYM, bn = (size_t)nb * p->bars_padded * SYM;
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) {
        if (full.a.out[k] && !(stored >> k & 1)) {
            nan_fill_kernel<<<e->sm_count * 4, 256, 0, e->stream>>>(full.a.out[k] + boff, bn);
            CU(cudaGetLastError());
            ++n_launch;
        }
    }
    // one launch of the fused kernel for the groups of `a` (variant selection + tail spreading)
    // nl blocks: the range [b0, b0 + nb) itself (list == nullptr) or the device list `list` of nl absolute block ids
    auto launch_one = [&](SuiteArgs a, const int *list, int64_t nl) -> int {
        const int64_t nb = nl;                                // (shadows the range length: variant selection goes by this launch)
        a.block0 = list ? 0 : (int)b0;
        a.blist = list;
        derive_roles(a);
        // CTA shape of a launch with few role warps per block (partial suites, optional groups): field-sized stages and the CTA
        // width with the fewest waves -- see the comment at the partial-suite launch below
        auto shape_few_warps = [&](const void *kernel, SuiteArgs &x, int n_slots, int &threads, int &smem) {
            static const bool slim = !getenv("PQB_BASE_SLIM") || atoi(getenv("PQB_BASE_SLIM")) != 0;
            static const int warps = getenv("PQB_BASE_WARPS") ? atoi(getenv("PQB_BASE_WARPS")) : 0;
            static const int min_smem = getenv("PQB_BASE_SMEM") ? atoi(getenv("PQB_BASE_SMEM")) : 0;
            int top = 0;
            for (int f = 0; f < N_IN; ++f) if (x.fields >> f & 1) top = f + 1;
            x.stage_stride = slim ? top * SB * SYM * 8 : STAGE_BYTES;
            smem = std::max(x.smem_bytes - NS * (STAGE_BYTES - x.stage_stride), min_smem);
            threads = CTA_THREADS;
            int occ = 0;
            if (warps > 0) threads = 32 * std::min(N_ROLES + 1, std::max(warps, n_slots + 1));
            else if (x.split_from < 0 && nb > 3ll * e->sm_count) {          // (up to three blocks per SM the eight-warp CTA is one wave already)
                int64_t best = INT64_MAX;
                for (int W = N_ROLES + 1; W > n_slots; --W) {
                    // (warp w runs on SM sub-partition w % 4: the producer -- the last warp, polling its mbarriers -- must not share
                    // one with a role warp while a sub-partition without one exists: KDJ + ATR with W = 6 took 3.76 ms, W = 8 2.96)
                    if (n_slots < 4 && (W - 1) % 4 < n_slots) continue;
                    if (W > 4 && W <= N_ROLES) continue;      // (5 - 7 warps measured erratic: WILLR + MIDPRICE 4.17 ms with 4 or 8 warps, 4.72 with 6)
                    int k = 0;
                    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k, kernel, 32 * W, (size_t)smem) != cudaSuccess || k <= 0) continue;
                    const int64_t waves = (nb + (int64_t)k * e->sm_count - 1) / ((int64_t)k * e->sm_count);
                    if (waves < best) { best = waves; threads = 32 * W; occ = k; }
                }
            }
            // Two-warp CTAs (one slot + the producer): the role warps of the resident CTAs all sat on two of the four SM sub-partitions (ncu, EMA
            // alone: one scheduler 95 % busy, the next 9 %) -- warp slots go to CTAs in pairs, so CTA j of an SM (blocks sm_count apart) swaps
            // role and producer warp when (j / 2) is odd (suite_kernel.cuh base_rot).  EMA alone 0.81 -> 0.72 ms (0.85 of peak), RSI 1.86 -> 1.31.
            // Wider CTAs: every rotation measured was slower (BBANDS, four warps: 1.68 -> 1.80 - 1.98 ms).  PQB_BASE_ROT=0: off
            static const int rot = getenv("PQB_BASE_ROT") ? atoi(getenv("PQB_BASE_ROT")) : 1;
            x.base_rot = (rot && x.split_from < 0 && threads == 64) ? e->sm_count : 0;
            x.base_rot_pair = 1;
            static const bool print_occ = getenv("PQB_PRINT_OCC") != nullptr;
            if (print_occ) {
                if (!occ) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, (size_t)smem);
                fprintf(stderr, "[pqb] few-warp launch: %d slots, %d threads, %d B smem -> %d CTAs per SM, %lld blocks\n", n_slots, threads, smem, occ, (long long)nb);
            }
        };
#if defined(PQB_DEBUG_CLOCKS) || defined(PQB_DEBUG_SMID)      // tuning builds: per-role busy cycles of the first block (costs ~18% on config 4) / the SM of every CTA
        if (!g_dbg) { CU(cudaMalloc(&g_dbg, 4096 * sizeof(unsigned long long))); CU(cudaMemset(g_dbg, 0xff, 4096 * sizeof(unsigned long long))); }
        a.dbg = g_dbg;
#else
        a.dbg = nullptr;
#endif
        bool fulls = a.gmask == G_ALL;                                       // exactly the benchmark suite
        for (int k = 0; k < PQB_N_SUITE_OUTPUTS; ++k) fulls &= a.out[k] != nullptr;
        const bool fastk = a.out[PQB_OUT_FASTK] != nullptr;                  // only the general / null-aware kernels store it
        fulls &= !fastk;
        // tail spreading: a FEW blocks beyond one CTA per SM (config 2: 157 blocks, 148 SMs) run as 7 single-role CTAs
        // each, which the block scheduler spreads over the SMs instead of doubling the load of a few of them
        // (0.838 -> 0.798 ms at config 2).  Only while every SM still holds at most two CTAs: each single-role CTA has
        // its own producer and stage ring, and beyond ~sm_count/7 extra blocks that costs more than it saves (measured:
        // 222 blocks split 1.41 ms, unsplit 0.84 ms).
        a.split_from = -1;
        unsigned grid = (unsigned)nb;
        const char *ts = getenv("PQB_TAIL_SPLIT");
        const bool tail_ok = !ts || atoi(ts) != 0;
        const char *ps = getenv("PQB_PIPELINE");
        const bool pipe_ok = !ps || atoi(ps) != 0;
        // the small-panel variant: nine role warps (two CTAs of 320 threads fit an SM)
        const bool small = fulls && pipe_ok && !a.vmask && a.mid_own && nb <= small_max_blocks(e);
        // a launch of optional groups only: the general kernel with its seven warps dealt as slots (suite_kernel.cuh)
        const char *ws = getenv("PQB_WIDE");
        const bool wide = !a.vmask && a.gmask && !(a.gmask & (unsigned)G_ALL) && (!ws || atoi(ws) != 0);
        const int nr = small ? N_ROLES_X : wide ? N_SLOTS_W : N_ROLES;
        int parts = nr;                                       // in-grid tail CTAs per split block (default: one role each)
        if (const char *tp = getenv("PQB_TAIL_PARTS")) if (!tail_compact()) parts = std::max(1, std::min(nr, atoi(tp)));
        a.split_parts = parts;
        a.split_compact = 0;
        if (tail_ok && nb > e->sm_count && nb <= e->sm_count + e->sm_count / nr && !(small && tail_compact())) {
            a.split_from = e->sm_count;
            grid = (unsigned)(e->sm_count + (nb - e->sm_count) * parts);
        }
        // tuning: PQB_SPLIT_ALL=<parts> splits EVERY block of a launch between one and two CTAs per SM into that many CTAs
        static const int split_all = getenv("PQB_SPLIT_ALL") ? atoi(getenv("PQB_SPLIT_ALL")) : 0;
        if (split_all > 1 && fulls && !small && nb > e->sm_count + e->sm_count / nr && nb < 2ll * e->sm_count) {
            a.split_from = 0;
            a.split_parts = std::min(nr, split_all);
            grid = (unsigned)(nb * a.split_parts);
        }
        if (a.vmask && fulls && a.nulls_fast && nulls_fulls()) suite_fused_kernel<true, true><<<grid, CTA_THREADS, a.smem_bytes, e->stream>>>(a);
        else if (a.vmask) suite_fused_kernel<false, true><<<grid, CTA_THREADS, a.smem_bytes, e->stream>>>(a);
        // small panels (about one CTA per SM) are bound by the length of each role's dependent FP64 chain per bar, not by
        // issue slots or HBM: they run the variant whose division-heavy roles (BBANDS, RSI, STOCH) are software-pipelined
        // over bars (suite_kernel.cuh "software-pipelined steady bar"); large panels are throughput-bound and run the
        // plain one (the pipelined loops execute more instructions)
        else if (small && tail_compact() && tail_ok && nb > e->sm_count) {
            // one whole-block CTA per SM; the blocks beyond run beside them as COMPACT tail CTAs (a launch of its own on a
            // second stream: `parts` CTAs per block, each 32 * (roles per CTA + 1) threads with its own producer and ring),
            // so a tail CTA holds 4 warps of registers instead of 10 and the block scheduler can put two of them next to a
            // whole-block CTA -- no SM walks two whole blocks
            const int cp = tail_parts_compact(e, nb - e->sm_count);
            SuiteArgs m = a, t = a;
            m.split_from = -1;
            t.split_from = 0; t.split_parts = cp; t.split_compact = 1;
            if (t.blist) t.blist += e->sm_count; else t.block0 += e->sm_count;
            const int roles_per_cta = (N_ROLES_X + cp - 1) / cp;
            CU(cudaEventRecord(e->ev_fork, e->stream));
            CU(cudaStreamWaitEvent(e->aux, e->ev_fork, 0));
            suite_fused_kernel<true, false, false, true><<<(unsigned)e->sm_count, CTA_THREADS_X, m.smem_bytes, e->stream>>>(m);
            suite_fused_kernel<true, false, false, true><<<(unsigned)((nb - e->sm_count) * cp), 32 * (roles_per_cta + 1), t.smem_bytes, e->aux>>>(t);
            CU(cudaEventRecord(e->ev_join, e->aux));
            CU(cudaStreamWaitEvent(e->stream, e->ev_join, 0));
            ++n_launch;
        }
        else if (small)
            suite_fused_kernel<true, false, false, true><<<grid, CTA_THREADS_X, a.smem_bytes, e->stream>>>(a);
        else if (fulls && force_base()) {                   // tuning: the partial-suite kernel (seven warps, pipelined roles) on the full suite
            deal_base_slots(a);
            a.stage_stride = STAGE_BYTES;
            suite_fused_kernel<false, false, true><<<grid, CTA_THREADS, a.smem_bytes, e->stream>>>(a);
        }
        else if (fulls) suite_fused_kernel<true, false><<<grid, CTA_THREADS, fulls_smem(a.smem_bytes), e->stream>>>(a);
        else if (!(a.gmask & ~(unsigned)G_ALL) && !fastk) {
            deal_base_slots(a);
            // A partial suite has few role warps per block, so an eight-warp CTA (three per SM by registers) leaves a large panel
            // latency-bound AND in many waves of equal serial walks (50,000 x 5,040, EMA alone: 4 waves of 0.31 ms).  Two measures
            // (profiles/r05_partial_suite_cta_shapes.txt): the TMA stages hold only the fields this launch reads (close alone: 2 KB
            // per stage instead of 8), and the CTA is launched with W warps, n_slots + 1 <= W <= 8 -- the W with the fewest waves,
            // the widest such (fewer co-resident walks are faster walks).  EMA 1.24 -> 0.81 ms, RSI 2.36 -> 1.85, BBANDS 2.10 -> 1.68.
            // tuning: PQB_BASE_SLIM=0 full-size stages, PQB_BASE_WARPS=W fixes the width (8 = as before), PQB_BASE_SMEM = dynamic
            // shared memory to ask for at least, PQB_PRINT_OCC=1 prints the choice
            int threads, smem;
            shape_few_warps((const void *)suite_fused_kernel<false, false, true>, a, a.n_roles, threads, smem);
            suite_fused_kernel<false, false, true><<<grid, threads, smem, e->stream>>>(a);
        }
        else if (wide) {
            int n_slots = 0, threads, smem;
            for (int s = 0; s < N_SLOTS_W; ++s) n_slots += (a.gmask & slot_mask_w(s)) ? 1 : 0;
            shape_few_warps((const void *)suite_fused_kernel<false, false, false, true>, a, n_slots, threads, smem);
            suite_fused_kernel<false, false, false, true><<<grid, threads, smem, e->stream>>>(a);
        }
        else suite_fused_kernel<false, false><<<grid, CTA_THREADS, a.smem_bytes, e->stream>>>(a);
        CU(cudaGetLastError());
        ++n_launch;
        return PQB_OK;
    };
    if (full.a.gmask) {
        // benchmark groups and optional groups together: two launches -- the benchmark groups through their
        // compile-time-specialised kernels (full suite / partial suite), the optional groups through the general one
        // (it re-reads the input planes; the general kernel is 2.4x slower on the benchmark groups than the full-suite
        // kernel: 50,000 x 5,040 suite + MOM 23.2 ms in one general launch).  The flagged blocks of a panel with nulls split the
        // same way, between two null-aware launches (launch_null below).
        const unsigned gb = full.a.gmask & (unsigned)G_ALL, go = full.a.gmask & ~(unsigned)G_ALL;
        int rc;
        // which blocks of the range need the null-aware kernel
        int64_t n_null = 0;
        if (p->nulls_mode)
            for (int64_t b = b0; b < b0 + nb; ++b) n_null += p->h_blk_null[(size_t)b];
        const int *plain_list = nullptr, *null_list = nullptr;
        // The benchmark suite's null-aware kernel (<FULLS, NULLS> with fast stages) walks a block with a few halted symbols about as fast
        // as the plain kernel does, so flagged blocks simply run through it, beside the plain launch: no gather, no write-back, no
        // scattered stores (50,000 x 5,040 with 5 % halted symbols: 22.8 ms compacted).  Symbol compaction stays for the launches that
        // kernel does not serve (partial suites).  PQB_NULLS_PREFER_DISPATCH=0: compact whenever the panel is prepared for it.
        static const bool prefer_dispatch = !getenv("PQB_NULLS_PREFER_DISPATCH") || atoi(getenv("PQB_NULLS_PREFER_DISPATCH")) != 0;
        bool fast_suite = prefer_dispatch && full.a.gmask == (unsigned)G_ALL && nulls_fast_ok(full.a) && nulls_fulls();
        for (int k = 0; k < PQB_N_SUITE_OUTPUTS; ++k) fast_suite &= full.a.out[k] != nullptr;
        // ... on a panel of several waves with more than a handful of flagged symbols.  A null-aware CTA that shares its SM with plain CTAs
        // in the latency regime walks 1.6x slower (8,192 x 5,040 with 83 halted symbols: 3.0 ms dispatched, 2.2 ms compacted onto SMs of
        // their own), and up to ~64 flagged symbols the gather / write-back is cheaper than a slower block per symbol (20,000 x 5,040:
        // 20 halted 5.5 ms compacted / 5.8 dispatched, 200 halted 6.2 / 5.2)
        // (beyond 1,024 flagged symbols compaction stores straight into the symbols' lanes -- scattered 8-byte stores, ~0.15 ms per compacted
        // block: there the dispatch wins on a small panel too; PQB_NULLS_DISPATCH_SMALL_FROM = that count)
        static const int small_from = getenv("PQB_NULLS_DISPATCH_SMALL_FROM") ? atoi(getenv("PQB_NULLS_DISPATCH_SMALL_FROM")) : 1024;
        // ... and whenever four blocks out of five hold a flagged symbol anyway (8,192 x 5,040 with 409 halted symbols, one per block or more:
        // 3.7 ms compacted, 2.25 ms with every block in the null-aware kernel)
        fast_suite = fast_suite && ((nb > 3ll * e->sm_count && p->n_x > 64) || p->n_x > small_from || n_null * 5 >= nb * 4);
        did_compact = p->compact && n_null && !go && b0 == 0 && nb == p->n_blocks && !fast_suite;
        if (did_compact) {
            // ---- symbol compaction: flagged symbols -> blocks of their own (null-aware kernel, second stream) while the plain
            //      kernel runs every original block; the flagged lanes are overwritten afterwards ----
            const int64_t n_xb = p->n_xblocks;
            CompactArgs G{};
            for (int f = 0; f < PQB_N_FIELDS; ++f)
                if (p->d_in[f] && p->x_in[f]) { G.src[G.n_planes] = p->d_in[f]; G.dst[G.n_planes] = p->x_in[f]; ++G.n_planes; }
            G.symmap = p->d_symmap; G.bars_padded = (int)p->bars_padded; G.n_slots = (int)(n_xb * SYM);
            compact_kernel<true><<<dim3((unsigned)(n_xb * SYM), (unsigned)((G.n_planes + 7) / 8)), 256, 0, e->stream>>>(G);
            CU(cudaGetLastError());
            ++n_launch;
            // (the plain launch below waits for an event recorded on the second stream right before the null-aware kernel: both
            // become eligible together, and the null-aware CTAs -- a ~6 ms walk -- must be placed before the plain grid fills the GPU)
            CU(cudaEventRecord(e->ev_fork, e->stream));
            CU(cudaStreamWaitEvent(e->aux, e->ev_fork, 0));
            CU(cudaEventRecord(e->ev_pre, e->aux));
            // Two modes.  OVERLAPPED (few flagged symbols): the null-aware kernel writes compacted output planes on the second stream
            // while the plain kernel runs, and a write-back pass (~3.6 us per symbol) puts the lanes in place.  DIRECT (many): the
            // null-aware kernel runs AFTER the plain one on the same stream and stores straight into the symbols' own lanes
            // (SuiteArgs::symmap), overwriting what the plain kernel left there -- no overlap, but no write-back either.
            static const int direct_from = getenv("PQB_COMPACT_DIRECT_FROM") ? atoi(getenv("PQB_COMPACT_DIRECT_FROM")) : 1024;
            const bool direct = p->n_x > direct_from;
            SuiteArgs an = full.a;
            an.nulls_fast = nulls_fast_ok(full.a);
            an.start = nullptr;
            an.vmask = p->x_vmask;
            an.symflags = p->d_xflags;
            for (int f = 0; f < PQB_N_FIELDS; ++f) an.in[f] = p->x_in[f];
            for (int k = 0; k < PQB_N_OUTPUTS; ++k) { an.ovm[k] = p->x_ovm[k]; an.out[k] = !full.a.out[k] ? nullptr : direct ? full.a.out[k] : p->x_out[k]; }
            an.symmap = direct ? p->d_symmap : nullptr;
            an.n_symbols = (int)p->n_x; an.n_blocks = (int)n_xb; an.block0 = 0; an.blist = nullptr;
            an.split_from = -1; an.split_parts = N_ROLES; an.split_compact = 0; an.dbg = nullptr;
            if (!an.smem_bytes && (rc = layout_rings(an, p))) return rc;
            derive_roles(an);
            // (exclusive: with the whole shared memory of an SM requested, no plain CTA can move in beside a null-aware CTA)
            static const int exclusive = getenv("PQB_COMPACT_EXCLUSIVE") ? atoi(getenv("PQB_COMPACT_EXCLUSIVE")) : 1;
            static const int split0 = getenv("PQB_COMPACT_SPLIT0") ? atoi(getenv("PQB_COMPACT_SPLIT0")) : 1;
            bool fulls_n = an.gmask == (unsigned)G_ALL && an.nulls_fast && nulls_fulls();
            for (int k = 0; k < PQB_N_SUITE_OUTPUTS; ++k) fulls_n &= an.out[k] != nullptr;
            auto launch_null = [&](cudaStream_t st) {
                if (fulls_n)                // (exactly the benchmark suite: the compile-time-specialised null-aware kernel)
                    suite_fused_kernel<true, true><<<(unsigned)n_xb, CTA_THREADS, exclusive ? kMaxSmem : an.smem_bytes, st>>>(an);
                else if (split0 && exclusive)    // (the variant with SMA / EMA / TEMA / MACD over two warps: 288 threads, one CTA per SM)
                    suite_fused_kernel<false, true, false, true><<<(unsigned)n_xb, CTA_THREADS + 32, kMaxSmem, st>>>(an);
                else
                    suite_fused_kernel<false, true><<<(unsigned)n_xb, CTA_THREADS, exclusive ? kMaxSmem : an.smem_bytes, st>>>(an);
                ++n_launch;
                return cudaGetLastError();
            };
            SuiteArgs ap = full.a;
            ap.start = p->d_start_c;
            if (direct) {
                if ((rc = launch_one(ap, nullptr, nb))) return rc;
                CU(launch_null(e->stream));
            } else {
                CU(launch_null(e->aux));
                CU(cudaEventRecord(e->ev_join, e->aux));
                static const int order = getenv("PQB_COMPACT_ORDER") ? atoi(getenv("PQB_COMPACT_ORDER")) : 0;
                if (order == 0) {
                    CU(cudaStreamWaitEvent(e->stream, e->ev_pre, 0));
                    static const int delay_us = getenv("PQB_COMPACT_DELAY_US") ? atoi(getenv("PQB_COMPACT_DELAY_US")) : 40;
                    if (delay_us > 0) { delay_kernel<<<1, 32, 0, e->stream>>>((unsigned)delay_us * 1000u); CU(cudaGetLastError()); }
                }
                if (order == 2) CU(cudaStreamWaitEvent(e->stream, e->ev_join, 0));  // (tuning: no overlap at all)
                if ((rc = launch_one(ap, nullptr, nb))) return rc;
                CU(cudaStreamWaitEvent(e->stream, e->ev_join, 0));
                CompactArgs Sc{};
                for (int k = 0; k < PQB_N_OUTPUTS; ++k)
                    if (full.a.out[k] && p->x_out[k] && (stored >> k & 1)) {
                        if (Sc.n_planes == N_OUT) break;
                        Sc.src[Sc.n_planes] = p->x_out[k]; Sc.dst[Sc.n_planes] = full.a.out[k]; ++Sc.n_planes;
                    }
                Sc.symmap = p->d_symmap; Sc.bars_padded = (int)p->bars_padded; Sc.n_slots = (int)(n_xb * SYM);
                compact_kernel<false><<<dim3((unsigned)(n_xb * SYM), (unsigned)((Sc.n_planes + 7) / 8)), 256, 0, e->stream>>>(Sc);
                CU(cudaGetLastError());
                ++n_launch;
            }
        } else
        if (n_null && n_null < nb) {
            if (!p->d_blist) CU(cudaMalloc(&p->d_blist, (size_t)p->n_blocks * 2 * sizeof(int)));
            if (p->h_blist.empty()) p->h_blist.assign((size_t)p->n_blocks * 2, 0);
            int *hp = p->h_blist.data() + b0, *hn = p->h_blist.data() + p->n_blocks + b0;
            int64_t np_ = 0, nn = 0;
            for (int64_t b = b0; b < b0 + nb; ++b) {
                if (p->h_blk_null[(size_t)b]) hn[nn++] = (int)b; else hp[np_++] = (int)b;
            }
            CU(cudaMemcpyAsync(p->d_blist + b0, hp, (size_t)np_ * sizeof(int), cudaMemcpyHostToDevice, e->stream));
            CU(cudaMemcpyAsync(p->d_blist + p->n_blocks + b0, hn, (size_t)nn * sizeof(int), cudaMemcpyHostToDevice, e->stream));
            plain_list = p->d_blist + b0;
            null_list = p->d_blist + p->n_blocks + b0;
        }
        // per-block dispatch with both kinds of blocks: the null-aware launch (the longer walk) goes first, on the second stream,
        // and the plain launch runs beside it (8,192 x 5,040 with one halted symbol: 1.6 + 1.9 ms back to back -> side by side)
        static const bool side_by_side = !getenv("PQB_NULLS_CONCURRENT") || atoi(getenv("PQB_NULLS_CONCURRENT")) != 0;
        // the flagged blocks.  Next to optional groups the benchmark groups keep a null-aware launch of their own -- the
        // specialised kernel with fast stages when all 21 suite outputs are bound, as without optional groups -- and the optional
        // groups, whose null rules have no fast stages, walk the same blocks through the general null-aware kernel.
        auto launch_null = [&]() -> int {
            if (gb && go && split_launch_enabled()) {
                SuiteArgs ab = null_variant(p, full.a), ao = ab;
                ab.gmask = gb;
                ab.steady_lead = full.steady_b;
                for (int k = 0; k < PQB_N_OUTPUTS; ++k) if (outputs_of_groups(go) >> k & 1) ab.out[k] = nullptr;
                ab.nulls_fast = nulls_fast_ok(ab);
                ao.gmask = go;
                if ((rc = layout_rings(ab, p)) || (rc = layout_rings(ao, p))) return rc;      // (subsets of a layout that fits)
                if ((rc = launch_one(ab, null_list, n_null))) return rc;
                return launch_one(ao, null_list, n_null);
            }
            SuiteArgs an = null_variant(p, full.a);
            if (!an.smem_bytes && (rc = layout_rings(an, p))) return rc;
            return launch_one(an, null_list, n_null);
        };
        bool null_done = false;
        if (!did_compact && n_null && n_null < nb && side_by_side) {
            CU(cudaEventRecord(e->ev_fork, e->stream));       // (after the block lists' copies)
            CU(cudaStreamWaitEvent(e->side, e->ev_fork, 0));
            std::swap(e->stream, e->side);                    // (a null-aware launch_one() touches e->stream only)
            rc = launch_null();
            std::swap(e->stream, e->side);
            if (rc) return rc;
            null_done = true;
        }
        if (!did_compact && n_null < nb) {                    // the plain blocks
            const int64_t nl = nb - n_null;
            if (gb && go && split_launch_enabled()) {
                SuiteArgs ab = full.a, ao = full.a;
                ab.gmask = gb;
                ao.gmask = go;
                if ((rc = layout_rings(ab, p)) || (rc = layout_rings(ao, p))) return rc;      // (subsets of a layout that fits)
                if ((rc = launch_one(ab, plain_list, nl))) return rc;
                if ((rc = launch_one(ao, plain_list, nl))) return rc;
            } else if ((rc = launch_one(full.a, plain_list, nl))) return rc;
        }
        if (null_done) {                                      // join the second stream
            CU(cudaEventRecord(e->ev_side, e->side));
            CU(cudaStreamWaitEvent(e->stream, e->ev_side, 0));
        } else if (!did_compact && n_null) {
            if ((rc = launch_null())) return rc;
        }
    }
#ifdef PQB_DEBUG_SMID
    if (g_dbg && full.a.gmask) {
        static unsigned long long h[4096];
        CU(cudaStreamSynchronize(e->stream));
        CU(cudaMemcpy(h, g_dbg, sizeof h, cudaMemcpyDeviceToHost));
        int whole[256] = {0}, part[256] = {0};
        for (int i = 0; i < 2048; ++i) if (h[i] < 256) ++whole[h[i]];
        for (int i = 2048; i < 4096; ++i) if (h[i] < 256) ++part[h[i]];
        int hist[8][8] = {{0}};
        for (int s = 0; s < e->sm_count; ++s) ++hist[std::min(whole[s], 7)][std::min(part[s], 7)];
        fprintf(stderr, "[pqb] SMs by (whole-block CTAs, tail CTAs):");
        for (int w = 0; w < 8; ++w) for (int t = 0; t < 8; ++t) if (hist[w][t]) fprintf(stderr, " (%d,%d)x%d", w, t, hist[w][t]);
        fprintf(stderr, "\n");
        CU(cudaMemset(g_dbg, 0xff, sizeof h));
    }
#endif
#ifdef PQB_DEBUG_CLOCKS
    if (g_dbg && full.a.gmask) {
        unsigned long long h[N_ROLES];
        CU(cudaStreamSynchronize(e->stream));
        CU(cudaMemcpy(h, g_dbg, sizeof h, cudaMemcpyDeviceToHost));
        fprintf(stderr, "[pqb] busy cycles/bar by role (block %lld):", (long long)b0);
        for (int r = 0; r < N_ROLES; ++r) fprintf(stderr, " r%d=%.0f", r, (double)h[r] / (double)p->n_bars);
        fprintf(stderr, "\n");
    }
#endif
    if (ev_after_fused) CU(cudaEventRecord(ev_after_fused, e->stream));
    const int64_t s0 = b0 * SYM, ns = std::min<int64_t>(nb * SYM, p->n_symbols - s0);
    int64_t n_null = 0;
    if (p->nulls_mode && !did_compact)
        for (int64_t b = b0; b < b0 + nb; ++b) n_null += p->h_blk_null[(size_t)b];
    // validity words written by a kernel -> Arrow bitmaps: outputs [k0, N) of the blocks `list` (or of the whole range)
    auto unpack_masks = [&](int k0, const int *list, int64_t nl, bool clear_unstored) -> int {
        MaskArgs M{};
        int n = 0;
        for (int k = k0; k < PQB_N_OUTPUTS; ++k) {
            if (!(full.a.out[k] && p->d_bits[k])) continue;
            if (stored >> k & 1) {
                M.tiled_in[n] = p->d_ovm[k];
                M.rm_out[n] = p->d_bits[k];
                ++n;
            } else if (clear_unstored) {
                CU(cudaMemsetAsync(p->d_bits[k] + (size_t)s0 * p->words_per_row, 0,
                                   (size_t)ns * p->words_per_row * sizeof(uint32_t), e->stream));
            }
        }
        if (!n || !nl) return PQB_OK;
        M.n_planes = n; M.n_symbols = (int)p->n_symbols; M.n_bars = (int)p->n_bars; M.bars_padded = (int)p->bars_padded;
        M.words_per_row = (int)p->words_per_row; M.n_blocks = (int)nl;
        M.block0 = (int)b0; M.blist = list;
        dim3 grid((unsigned)p->words_per_row, (unsigned)nl);
        unpack_mask_kernel<<<grid, 32, 0, e->stream>>>(M);
        CU(cudaGetLastError());
        ++n_launch;
        return PQB_OK;
    };
    if (n_null == nb) {
        // every block of the range ran the null-aware kernel: all validity comes from its per-bar words
        int rc = unpack_masks(0, nullptr, nb, true);
        if (launches) *launches = n_launch;
        return rc;
    }
    {   // optional groups: validity words written by the kernel (or all-null for a period-0 column)
        int rc = unpack_masks(PQB_N_SUITE_OUTPUTS, nullptr, nb, true);
        if (rc) return rc;
    }
    ValidityArgs V{};
    bool any = false;
    for (int k = 0; k < PQB_N_OUTPUTS; ++k) {
        V.bits[k] = (k < PQB_N_SUITE_OUTPUTS && full.a.out[k] && p->d_bits[k]) ? p->d_bits[k] + (size_t)s0 * p->words_per_row : nullptr;
        V.lead[k] = full.lead[k];
        any |= V.bits[k] != nullptr;
    }
    V.start = did_compact ? p->d_start_c : full.a.start ? full.a.start + s0 : nullptr;
    V.n_symbols = (int)ns;
    V.n_bars = full.a.n_bars;
    V.words_per_row = (int)p->words_per_row;
    if (any) {
        const long long total = (long long)V.n_symbols * V.words_per_row;
        const int grid = (int)std::min<long long>((total + 255) / 256, (long long)e->sm_count * 8);
        validity_kernel<<<grid, 256, 0, e->stream>>>(V);
        CU(cudaGetLastError());
        ++n_launch;
    }
    if (n_null) {
        // mixed range: the flagged blocks' bitmaps come from the null-aware kernel's words (overwriting the lead-based ones)
        int rc = unpack_masks(0, p->d_blist + p->n_blocks + b0, n_null, false);
        if (rc) return rc;
    }
    if (did_compact) {
        // the flagged symbols' bitmaps from the compacted blocks' validity words, row by row through the slot -> symbol map
        MaskArgs M{};
        int n = 0;
        for (int k = 0; k < PQB_N_OUTPUTS; ++k)
            if (full.a.out[k] && p->d_bits[k] && p->x_ovm[k] && (stored >> k & 1)) { M.tiled_in[n] = p->x_ovm[k]; M.rm_out[n] = p->d_bits[k]; ++n; }
        if (n) {
            M.n_planes = n; M.n_symbols = (int)p->n_symbols; M.n_bars = (int)p->n_bars; M.bars_padded = (int)p->bars_padded;
            M.words_per_row = (int)p->words_per_row; M.n_blocks = (int)p->n_xblocks; M.block0 = 0; M.blist = nullptr;
            M.symmap = p->d_symmap;
            dim3 grid((unsigned)p->words_per_row, (unsigned)p->n_xblocks);
            unpack_mask_kernel<<<grid, 32, 0, e->stream>>>(M);
            CU(cudaGetLastError());
            ++n_launch;
        }
    }
    if (launches) *launches = n_launch;
    return PQB_OK;
}

// the optional groups report validity per bar: allocate their validity-word planes on first use
static int ensure_extra_masks(pqb_panel *p, const pqb_suite_params *sp) {
    if (!(sp->indicators & (PQB_IND_EXTRAS | PQB_IND_FASTK))) return PQB_OK;
    const size_t mwords = (size_t)p->n_blocks * p->bars_padded;
    for (int k = PQB_N_SUITE_OUTPUTS; k < PQB_N_OUTPUTS; ++k)
        if (p->d_out[k] && !p->d_ovm[k]) CU(cudaMalloc(&p->d_ovm[k], mwords * sizeof(uint32_t)));
    return PQB_OK;
}

static int run_suite(pqb_panel *p, const pqb_suite_params *sp, cudaEvent_t ev_after_fused, int *launches) {
    if (!p || !sp) return fail(PQB_ERR_INVALID, "pqb_suite_run: NULL argument");
    int rc = set_dev(p->e);
    if (rc) return rc;
    if ((rc = ensure_extra_masks(p, sp))) return rc;
    Built b;
    if ((rc = build_args(p, sp, &b))) return rc;
    int nl = 0;
    rc = launch_suite(p, b, 0, p->n_blocks, ev_after_fused, &nl);
    p->last_launches = nl;
    if (launches) *launches = nl;
    return rc;
}

extern "C" int pqb_suite_run(pqb_panel *p, const pqb_suite_params *sp) { return run_suite(p, sp, nullptr, nullptr); }

// ---------------------------------------------------------------------------------------
// end-to-end host path: per chunk of symbol blocks
//   h2d stream : pinned row-major fields -> device row-major buffer [c % 2]
//   compute    : pack -> fused suite -> validity -> unpack into device row-major buffer [c % 2]
//   d2h stream : outputs + bitmaps -> pinned staging
// so both DMA directions overlap the kernels of neighbouring chunks.
// ---------------------------------------------------------------------------------------
struct IntakeGate;
static void intake_wait(const IntakeGate *g, int64_t chunk);
static int run_host_impl(pqb_panel *p, const pqb_suite_params *sp, int64_t chunk_symbols, const IntakeGate *gate) {
    if (!p || !sp) return fail(PQB_ERR_INVALID, "pqb_suite_run_host: NULL argument");
    if (!p->staging) return fail(PQB_ERR_INVALID, "pqb_suite_run_host: panel has no host staging");
    int rc = set_dev(p->e);
    if (rc) return rc;
    pqb_engine *e = p->e;
    Built full;
    if ((rc = ensure_extra_masks(p, sp))) return rc;
    if ((rc = build_args(p, sp, &full))) return rc;
    if (chunk_symbols <= 0 || chunk_symbols > p->chunk_symbols) chunk_symbols = p->chunk_symbols;
    chunk_symbols = std::max<int64_t>(SYM, chunk_symbols / SYM * SYM);
    const int64_t n_chunks = (p->n_symbols + chunk_symbols - 1) / chunk_symbols;
    const size_t cplane = (size_t)p->chunk_symbols * p->pitch;
    Events up((size_t)n_chunks), done((size_t)n_chunks);
    CU(up.create(cudaEventDisableTiming));
    CU(done.create(cudaEventDisableTiming));
    // null bookkeeping -> device: the whole panel up front, or (pipelined intake) chunk by chunk as the columns arrive
    if (!gate && (rc = prepare_nulls(p, e->h2d))) return rc;
    int total_launches = 0;
    for (int64_t c = 0; c < n_chunks; ++c) {
        const int b = (int)(c & 1);
        const int64_t s0 = c * chunk_symbols, ns = std::min(chunk_symbols, p->n_symbols - s0);
        const size_t rows = (size_t)ns * p->pitch * sizeof(double);
        if (gate) {
            intake_wait(gate, c);
            if ((rc = prepare_nulls(p, e->h2d, s0, ns))) return rc;
        }
        // ---- H2D (buffer b is free once the pack of chunk c-2 has read it) ----
        if (c >= 2) CU(cudaStreamWaitEvent(e->h2d, p->ev_packed[b], 0));
        const double *rm_in[PQB_N_FIELDS];
        double *tl_in[PQB_N_FIELDS];
        int n_in = 0;
        for (int f = 0; f < PQB_N_FIELDS; ++f) {
            if (!p->d_in[f]) continue;
            double *buf = p->d_xin[b] + cplane * p->in_slot[f];
            CU(cudaMemcpyAsync(buf, p->h_in[f] + (size_t)s0 * p->pitch, rows, cudaMemcpyHostToDevice, e->h2d));
            rm_in[n_in] = buf; tl_in[n_in] = p->d_in[f]; ++n_in;
        }
        CU(cudaEventRecord(up[(size_t)c], e->h2d));
        // ---- compute ----
        CU(cudaStreamWaitEvent(e->stream, up[(size_t)c], 0));
        if ((rc = launch_conv(p, true, rm_in, tl_in, n_in, s0, ns, e->stream))) return rc;
        CU(cudaEventRecord(p->ev_packed[b], e->stream));
        int nl = 0;
        if ((rc = launch_suite(p, full, s0 / SYM, (ns + SYM - 1) / SYM, nullptr, &nl))) return rc;
        total_launches += nl + (n_in ? 1 : 0);
        if (c >= 2) CU(cudaStreamWaitEvent(e->stream, p->ev_d2h[b], 0));
        const double *rm_out[PQB_N_OUTPUTS];
        double *tl_out[PQB_N_OUTPUTS];
        double *host_out[PQB_N_OUTPUTS];
        int n_out = 0;
        for (int k = 0; k < PQB_N_OUTPUTS; ++k) {
            if (!full.a.out[k]) continue;
            rm_out[n_out] = p->d_xout[b] + cplane * p->out_slot[k]; tl_out[n_out] = p->d_out[k]; host_out[n_out] = p->h_out[k];
            ++n_out;
        }
        if ((rc = launch_conv(p, false, rm_out, tl_out, n_out, s0, ns, e->stream))) return rc;
        total_launches += n_out ? 1 : 0;
        CU(cudaEventRecord(done[(size_t)c], e->stream));
        // ---- D2H ----
        CU(cudaStreamWaitEvent(e->d2h, done[(size_t)c], 0));
        for (int i = 0; i < n_out; ++i)
            CU(cudaMemcpyAsync(host_out[i] + (size_t)s0 * p->pitch, rm_out[i], rows, cudaMemcpyDeviceToHost, e->d2h));
        const size_t boff = (size_t)s0 * p->words_per_row, bbytes = (size_t)ns * p->words_per_row * sizeof(uint32_t);
        for (int k = 0; k < PQB_N_OUTPUTS; ++k)
            if (full.a.out[k]) CU(cudaMemcpyAsync(p->h_bits[k] + boff, p->d_bits[k] + boff, bbytes, cudaMemcpyDeviceToHost, e->d2h));
        CU(cudaEventRecord(p->ev_d2h[b], e->d2h));
    }
    CU(cudaStreamSynchronize(e->d2h));
    CU(cudaStreamSynchronize(e->stream));
    CU(cudaStreamSynchronize(e->h2d));
    p->last_launches = total_launches;
    p->inputs_resident = true;
    return PQB_OK;
}

extern "C" int pqb_suite_run_host(pqb_panel *p, const pqb_suite_params *sp, int64_t chunk_symbols) {
    return run_host_impl(p, sp, chunk_symbols, nullptr);
}

extern "C" int pqb_panel_last_launches(const pqb_panel *p) { return p ? p->last_launches : 0; }

// ---------------------------------------------------------------------------------------
// measurement helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9e3779b97f4a7c15ULL;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}
// approx N(0,1): Irwin-Hall sum of 12 uniforms built from 6 hashes (2 x 32-bit halves each)
__device__ __forceinline__ double gauss(uint64_t key) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const uint64_t h = mix64(key * 6 + i);
        s += (double)(uint32_t)h * (1.0 / 4294967296.0) + (double)(uint32_t)(h >> 32) * (1.0 / 4294967296.0);
    }
    return s - 6.0;
}

// Synthetic random-walk OHLCV (SURVEY.md 8d) written straight into the tiled planes: one lane per
// symbol walks its row; a warp writes 256 B contiguous per plane per bar.
__global__ void __launch_bounds__(32) synth_kernel(double *c, double *h, double *l, double *v, int n_symbols,
                                                   int n_bars, int bars_padded, uint64_t seed, double sigma) {
    const int lane = threadIdx.x;
    const int s = blockIdx.x * SYM + lane;
    const size_t base = (size_t)blockIdx.x * bars_padded * SYM + lane;
    double close = 100.0;
    for (int t = 0; t < bars_padded; ++t) {
        const uint64_t key = (seed + (uint64_t)s) * 0x100000001b3ULL + (uint64_t)t * 4;
        const double open = close;
        close = open * exp(sigma * gauss(key));
        const double hi = fmax(open, close) * (1.0 + fabs(0.5 * sigma * gauss(key + 1)));
        const double lo = fmin(open, close) * (1.0 - fabs(0.5 * sigma * gauss(key + 2)));
        const double vol = rint(exp(13.0 + gauss(key + 3)));
        const bool live = t < n_bars && s < n_symbols;
        const size_t o = base + (size_t)t * SYM;
        if (c) c[o] = live ? close : 0.0;
        if (h) h[o] = live ? hi : 0.0;
        if (l) l[o] = live ? lo : 0.0;
        if (v) v[o] = live ? vol : 0.0;
    }
}

extern "C" int pqb_panel_fill_synthetic(pqb_panel *p, uint64_t seed, double sigma, int to_host) {
    if (!p) return fail(PQB_ERR_INVALID, "pqb_panel_fill_synthetic: NULL");
    int rc = set_dev(p->e);
    if (rc) return rc;
    synth_kernel<<<(unsigned)p->n_blocks, 32, 0, p->e->stream>>>(p->d_in[PQB_CLOSE], p->d_in[PQB_HIGH], p->d_in[PQB_LOW],
                                                                  p->d_in[PQB_VOLUME], (int)p->n_symbols, (int)p->n_bars,
                                                                  (int)p->bars_padded, seed, sigma);
    CU(cudaGetLastError());
    p->inputs_resident = true;
    if (to_host && p->staging && (rc = download_planes(p, true))) return rc;
    CU(cudaStreamSynchronize(p->e->stream));
    return PQB_OK;
}

extern "C" int pqb_suite_time(pqb_panel *p, const pqb_suite_params *sp, int warmup, int iters, float *ms_total,
                              float *ms_fused, int *launches_per_step) {
    if (!p || !sp || iters <= 0) return fail(PQB_ERR_INVALID, "pqb_suite_time: bad argument");
    int rc = set_dev(p->e);
    if (rc) return rc;
    cudaStream_t st = p->e->stream;
    int nl = 0;
    for (int i = 0; i < warmup; ++i)
        if ((rc = run_suite(p, sp, nullptr, &nl))) return rc;
    CU(cudaStreamSynchronize(st));
    Events b((size_t)iters), a((size_t)iters), e01(2);
    CU(b.create());
    CU(a.create());
    CU(e01.create());
    cudaEvent_t e0 = e01[0], e1 = e01[1];
    CU(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; ++i) {
        CU(cudaEventRecord(b[(size_t)i], st));
        if ((rc = run_suite(p, sp, a[(size_t)i], &nl))) return rc;
    }
    CU(cudaEventRecord(e1, st));
    CU(cudaStreamSynchronize(st));
    float tot = 0.f, fused = 0.f;
    CU(cudaEventElapsedTime(&tot, e0, e1));
    for (int i = 0; i < iters; ++i) {
        float t = 0.f;
        CU(cudaEventElapsedTime(&t, b[(size_t)i], a[(size_t)i]));
        fused += t;
    }
    if (ms_total) *ms_total = tot;
    if (ms_fused) *ms_fused = fused;
    if (launches_per_step) *launches_per_step = nl;
    return PQB_OK;
}

extern "C" int pqb_suite_time_host(pqb_panel *p, const pqb_suite_params *sp, int64_t chunk_symbols, int warmup,
                                   int iters, float *ms_total) {
    if (!p || !sp || iters <= 0) return fail(PQB_ERR_INVALID, "pqb_suite_time_host: bad argument");
    int rc = set_dev(p->e);
    if (rc) return rc;
    for (int i = 0; i < warmup; ++i)
        if ((rc = pqb_suite_run_host(p, sp, chunk_symbols))) return rc;
    // the whole pipeline spans three streams; bracket it with device-wide syncs and events on the
    // first / last stream of the pipeline
    Events e01(2);
    CU(e01.create());
    cudaEvent_t e0 = e01[0], e1 = e01[1];
    CU(cudaDeviceSynchronize());
    CU(cudaEventRecord(e0, p->e->h2d));
    for (int i = 0; i < iters; ++i)
        if ((rc = pqb_suite_run_host(p, sp, chunk_symbols))) return rc;
    CU(cudaEventRecord(e1, p->e->d2h));
    CU(cudaEventSynchronize(e1));
    float tot = 0.f;
    CU(cudaEventElapsedTime(&tot, e0, e1));
    if (ms_total) *ms_total = tot;
    return PQB_OK;
}

__global__ void flush_kernel(uint4 *p, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = make_uint4((unsigned)i, 1u, 2u, 3u);
}
// ---- measurement helper: what HBM delivers for a given read : write mix, without any indicator arithmetic ----
// A grid-stride kernel reads `n_reads` planes and writes `n_writes` planes with the suite's own 256-byte warp rows
// (streaming loads / stores).  bench.py runs it with the suite's mix (4 reads, 21 writes) next to the fused kernel:
// the copy bandwidth in MEASURED_PEAKS.json is a 1 : 1 mix, and a write-heavy mix gets less out of HBM3e.
struct MixArgs { const double *in[PQB_N_FIELDS]; double *out[PQB_N_OUTPUTS]; int n_in, n_out; };
__global__ void __launch_bounds__(256) stream_mix_kernel(const __grid_constant__ MixArgs P, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double s = 0.0;
        for (int f = 0; f < P.n_in; ++f) s += __ldcs(P.in[f] + i);
        for (int k = 0; k < P.n_out; ++k) __stcs(P.out[k] + i, s + (double)k);
    }
}

extern "C" int pqb_probe_pcie(pqb_engine *e, int64_t bytes, int iters, double gbs[4]) {
    if (!e || !gbs || bytes < (1 << 20) || iters < 1) return fail(PQB_ERR_INVALID, "pqb_probe_pcie: bad argument");
    int rc = set_dev(e);
    if (rc) return rc;
    const size_t out_b = (size_t)bytes, in_b = (size_t)bytes * 4 / 21 / 256 * 256;
    void *h_out = nullptr, *h_in = nullptr, *d_out = nullptr, *d_in = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    auto release = [&]() {
        if (h_out) host_give(e, h_out, out_b);
        if (h_in) host_give(e, h_in, in_b);
        if (d_out) cudaFree(d_out);
        if (d_in) cudaFree(d_in);
        for (auto &x : ev) if (x) cudaEventDestroy(x);
    };
    cudaError_t ce = host_take(e, &h_out, out_b);
    if (ce == cudaSuccess) ce = host_take(e, &h_in, in_b);
    if (ce == cudaSuccess) ce = cudaMalloc(&d_out, out_b);
    if (ce == cudaSuccess) ce = cudaMalloc(&d_in, in_b);
    for (auto &x : ev) if (ce == cudaSuccess) ce = cudaEventCreate(&x);
    if (ce != cudaSuccess) { release(); cudaGetLastError(); return fail(PQB_ERR_ALLOC, "pqb_probe_pcie: %s", cudaGetErrorString(ce)); }
    memset(h_in, 0, in_b);
    cudaMemsetAsync(d_out, 0, out_b, e->d2h);
    auto down = [&]() { return cudaMemcpyAsync(h_out, d_out, out_b, cudaMemcpyDeviceToHost, e->d2h); };
    auto up = [&]() { return cudaMemcpyAsync(d_in, h_in, in_b, cudaMemcpyHostToDevice, e->h2d); };
    down(); up();                                          // touch everything once
    cudaStreamSynchronize(e->d2h); cudaStreamSynchronize(e->h2d);
    float ms = 0.f;
    cudaEventRecord(ev[0], e->d2h);
    for (int i = 0; i < iters; ++i) down();
    cudaEventRecord(ev[1], e->d2h);
    cudaEventSynchronize(ev[1]);
    cudaEventElapsedTime(&ms, ev[0], ev[1]);
    gbs[0] = (double)out_b * iters / (ms * 1e-3) / 1e9;
    cudaEventRecord(ev[2], e->h2d);
    for (int i = 0; i < iters; ++i) up();
    cudaEventRecord(ev[3], e->h2d);
    cudaEventSynchronize(ev[3]);
    cudaEventElapsedTime(&ms, ev[2], ev[3]);
    gbs[1] = (double)in_b * iters / (ms * 1e-3) / 1e9;
    cudaEventRecord(ev[0], e->d2h);
    cudaEventRecord(ev[2], e->h2d);
    for (int i = 0; i < iters; ++i) { down(); up(); }
    cudaEventRecord(ev[1], e->d2h);
    cudaEventRecord(ev[3], e->h2d);
    cudaEventSynchronize(ev[1]);
    cudaEventSynchronize(ev[3]);
    cudaEventElapsedTime(&ms, ev[0], ev[1]);
    gbs[2] = (double)out_b * iters / (ms * 1e-3) / 1e9;
    cudaEventElapsedTime(&ms, ev[2], ev[3]);
    gbs[3] = (double)in_b * iters / (ms * 1e-3) / 1e9;
    ce = cudaGetLastError();
    release();
    if (ce != cudaSuccess) return fail(PQB_ERR_CUDA, "pqb_probe_pcie: %s", cudaGetErrorString(ce));
    return PQB_OK;
}

extern "C" int pqb_stream_mix(pqb_engine *e, int n_reads, int n_writes, int64_t doubles_per_plane, int warmup, int iters,
                              float *ms_per_iter) {
    if (!e || !ms_per_iter || n_reads < 0 || n_reads > PQB_N_FIELDS || n_writes < 1 || n_writes > PQB_N_OUTPUTS ||
        doubles_per_plane < 1 || iters < 1)
        return fail(PQB_ERR_INVALID, "pqb_stream_mix: bad argument");
    int rc = set_dev(e);
    if (rc) return rc;
    MixArgs P{};
    P.n_in = n_reads; P.n_out = n_writes;
    const size_t bytes = (size_t)doubles_per_plane * sizeof(double);
    std::vector<void *> owned;
    auto release = [&]() { for (void *q : owned) cudaFree(q); };
    cudaError_t ce = cudaSuccess;
    for (int f = 0; f < n_reads && ce == cudaSuccess; ++f) {
        void *q = nullptr;
        if ((ce = cudaMalloc(&q, bytes)) == cudaSuccess) { owned.push_back(q); P.in[f] = (const double *)q; ce = cudaMemsetAsync(q, 0, bytes, e->stream); }
    }
    for (int k = 0; k < n_writes && ce == cudaSuccess; ++k) {
        void *q = nullptr;
        if ((ce = cudaMalloc(&q, bytes)) == cudaSuccess) { owned.push_back(q); P.out[k] = (double *)q; }
    }
    cudaEvent_t a = nullptr, b = nullptr;
    if (ce == cudaSuccess) ce = cudaEventCreate(&a);
    if (ce == cudaSuccess) ce = cudaEventCreate(&b);
    const unsigned grid = (unsigned)e->sm_count * 8;
    for (int i = 0; i < warmup && ce == cudaSuccess; ++i) { stream_mix_kernel<<<grid, 256, 0, e->stream>>>(P, (size_t)doubles_per_plane); ce = cudaGetLastError(); }
    if (ce == cudaSuccess) ce = cudaEventRecord(a, e->stream);
    for (int i = 0; i < iters && ce == cudaSuccess; ++i) { stream_mix_kernel<<<grid, 256, 0, e->stream>>>(P, (size_t)doubles_per_plane); ce = cudaGetLastError(); }
    if (ce == cudaSuccess) ce = cudaEventRecord(b, e->stream);
    if (ce == cudaSuccess) ce = cudaEventSynchronize(b);
    float ms = 0.f;
    if (ce == cudaSuccess) ce = cudaEventElapsedTime(&ms, a, b);
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
    release();
    if (ce != cudaSuccess) { cudaGetLastError(); return fail(ce == cudaErrorMemoryAllocation ? PQB_ERR_ALLOC : PQB_ERR_CUDA, "pqb_stream_mix: %s", cudaGetErrorString(ce)); }
    *ms_per_iter = ms / (float)iters;
    return PQB_OK;
}

extern "C" int pqb_flush_l2(pqb_engine *e) {
    if (!e) return fail(PQB_ERR_INVALID, "pqb_flush_l2: NULL");
    int rc = set_dev(e);
    if (rc) return rc;
    if (!e->flush_buf) {
        e->flush_bytes = 256ull << 20;   // 2x the 126 MB L2
        CU(cudaMalloc(&e->flush_buf, e->flush_bytes));
    }
    flush_kernel<<<e->sm_count * 4, 256, 0, e->stream>>>((uint4 *)e->flush_buf, e->flush_bytes / 16);
    CU(cudaGetLastError());
    return PQB_OK;
}

extern "C" int pqb_selftest_divsqrt(pqb_engine *e, const double *a, const double *b, int64_t n, uint64_t result[4]) {
    if (!e || !a || !b || !result || n <= 0) return fail(PQB_ERR_INVALID, "pqb_selftest_divsqrt: bad arguments");
    int rc = set_dev(e);
    if (rc) return rc;
    double *da = nullptr, *db = nullptr;
    unsigned long long *dr = nullptr;
    CU(cudaMalloc(&da, n * sizeof(double)));
    CU(cudaMalloc(&db, n * sizeof(double)));
    CU(cudaMalloc(&dr, 4 * sizeof(unsigned long long)));
    CU(cudaMemcpyAsync(da, a, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemcpyAsync(db, b, n * sizeof(double), cudaMemcpyHostToDevice, e->stream));
    CU(cudaMemsetAsync(dr, 0, 4 * sizeof(unsigned long long), e->stream));
    divsqrt_selftest_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(da, db, n, dr);
    CU(cudaGetLastError());
    unsigned long long hr[4];
    CU(cudaMemcpyAsync(hr, dr, sizeof(hr), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < 4; ++i) result[i] = hr[i];
    cudaFree(da);
    cudaFree(db);
    cudaFree(dr);
    return PQB_OK;
}

// ---------------------------------------------------------------------------------------
// single-column entry points: one reference plugin call on one column
// ---------------------------------------------------------------------------------------
struct ColCheck { bool any_null; };
static ColCheck scan_col(const pqb_col *c) {
    ColCheck r{false};
    if (!c->validity) return r;
    for (int64_t i = 0; i < c->len; ++i)
        if (!bit_at(c->validity, c->offset + i)) { r.any_null = true; break; }
    return r;
}

enum NullPolicy { NP_SHIFT, NP_ERR };   // overlap/volatility/volume functions skip nulls; momentum.rs errors

static int run_single(pqb_engine *e, const pqb_col *const *cols, const int *fields, int n_cols, NullPolicy np,
                      const pqb_suite_params *sp, const int *outs, pqb_out_col *const *dst, int n_out) {
    if (!e) return fail(PQB_ERR_INVALID, "NULL engine");
    for (int i = 0; i < n_cols; ++i)
        if (!cols[i] || (!cols[i]->values && cols[i]->len > 0) || cols[i]->len < 0 || cols[i]->offset < 0)
            return fail(PQB_ERR_INVALID, "bad input column %d", i);
    for (int i = 0; i < n_out; ++i)
        if (!dst[i] || (!dst[i]->values && cols[0]->len > 0) || (!dst[i]->validity && cols[0]->len > 0))
            return fail(PQB_ERR_INVALID, "bad output column %d", i);
    const int64_t n = cols[0]->len;
    for (int i = 1; i < n_cols; ++i)
        if (cols[i]->len != n) return fail(PQB_ERR_INVALID, "input columns differ in length");
    for (int i = 0; i < n_cols; ++i) {
        ColCheck cc = scan_col(cols[i]);
        if (cc.any_null && np == NP_ERR)
            return fail(PQB_ERR_NULLS, "chunked array is not contiguous (input %d has nulls; reference: cont_slice()?)", i);
    }
    if (n == 0) return PQB_OK;
    // device required from here on
    int rc = set_dev(e);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(e->mu);
    if (!e->scratch || e->scratch_bars != n) {
        // park the current scratch, look for one of this length among the last few, else create it
        // (short columns only: a one-symbol panel of 1,000,000 bars holds 0.4 GB of pinned memory)
        if (e->scratch && e->scratch_bars <= 131072) e->scratch_lru.insert(e->scratch_lru.begin(), {e->scratch_bars, e->scratch});
        else if (e->scratch) pqb_panel_destroy(e->scratch);
        e->scratch = nullptr;
        for (size_t i = 0; i < e->scratch_lru.size(); ++i)
            if (e->scratch_lru[i].first == n) { e->scratch = e->scratch_lru[i].second; e->scratch_lru.erase(e->scratch_lru.begin() + (long)i); break; }
        while (e->scratch_lru.size() > 3) { pqb_panel_destroy(e->scratch_lru.back().second); e->scratch_lru.pop_back(); }
        if (!e->scratch) {
            rc = pqb_panel_create(e, 1, n, (1u << PQB_N_FIELDS) - 1, (1ull << PQB_N_OUTPUTS) - 1, 1, &e->scratch);
            if (rc) return rc;
        }
        e->scratch_bars = n;
    }
    pqb_panel *p = e->scratch;
    p->h_start_explicit[0] = 0;
    p->h_flags[0] = 0;
    for (int f = 0; f < PQB_N_FIELDS; ++f) { p->h_lead[f][0] = -1; p->h_vin[f].clear(); }
    uint32_t fmask = 0;
    for (int i = 0; i < n_cols; ++i) {
        if ((rc = pqb_panel_set_column(p, 0, fields[i], cols[i]->values, cols[i]->validity, cols[i]->offset, n))) return rc;
        fmask |= 1u << fields[i];
    }
    // only what this call touches crosses PCIe: the given fields up, the requested outputs down (the scratch panel has
    // every plane allocated; one EMA on a 1 M-bar column used to move 43 result planes)
    cudaStream_t st = e->stream;
    // short columns: no copy engine at all -- the pack kernel reads the pinned staging through its mapping and carries the
    // start, the unpack kernel writes values and validity words straight into the pinned result planes (a 2 KB column paid
    // ~12 us per cudaMemcpyAsync, 4 - 8 of them per call: EMA 104 us, MACD / BBANDS 165 us).  PQB_SINGLE_MAPPED = largest such
    // column in bars (0: always the copy engine)
    static const int64_t mapped_max = getenv("PQB_SINGLE_MAPPED") ? atoll(getenv("PQB_SINGLE_MAPPED")) : 32768;
    const bool mapped = n <= mapped_max && n_out <= CONV_MAX_BITS;
    if (mapped) {
        const double *rm[PQB_N_FIELDS];
        double *tl[PQB_N_FIELDS];
        int nf = 0;
        for (int f = 0; f < PQB_N_FIELDS; ++f)
            if (fmask >> f & 1) { rm[nf] = p->h_in[f]; tl[nf] = p->d_in[f]; ++nf; }
        const bool any_null = prepare_nulls_host(p, 0, 1);
        ConvArgs X{};
        X.start_dst = p->d_start; X.start_val = p->h_start[0];
        if ((rc = launch_conv(p, true, rm, tl, nf, 0, 1, st, &X))) return rc;
        p->inputs_resident = true;
        if ((rc = prepare_nulls_device(p, st, 0, 1, any_null, false))) return rc;
    } else {
        const double *rm[PQB_N_FIELDS];
        double *tl[PQB_N_FIELDS];
        int nf = 0;
        const size_t cplane = (size_t)p->chunk_symbols * p->pitch;
        for (int f = 0; f < PQB_N_FIELDS; ++f) {
            if (!(fmask >> f & 1)) continue;
            double *buf = p->d_xin[0] + cplane * p->in_slot[f];
            CU(cudaMemcpyAsync(buf, p->h_in[f], (size_t)p->pitch * sizeof(double), cudaMemcpyHostToDevice, st));
            rm[nf] = buf; tl[nf] = p->d_in[f]; ++nf;
        }
        if ((rc = launch_conv(p, true, rm, tl, nf, 0, 1, st))) return rc;
        p->inputs_resident = true;
        if ((rc = prepare_nulls(p, st))) return rc;
    }
    if ((rc = pqb_suite_run(p, sp))) return rc;
    if (mapped) {
        const double *rm[PQB_N_OUTPUTS];
        double *tl[PQB_N_OUTPUTS];
        ConvArgs X{};
        for (int i = 0; i < n_out; ++i) {
            rm[i] = p->h_out[outs[i]]; tl[i] = p->d_out[outs[i]];
            X.bits_src[i] = p->d_bits[outs[i]]; X.bits_dst[i] = p->h_bits[outs[i]];
        }
        X.n_bits = n_out; X.bits_words = (int)p->words_per_row;
        if ((rc = launch_conv(p, false, rm, tl, n_out, 0, 1, st, &X))) return rc;
    } else {
        const double *rm[PQB_N_OUTPUTS];
        double *tl[PQB_N_OUTPUTS];
        const size_t cplane = (size_t)p->chunk_symbols * p->pitch;
        for (int i = 0; i < n_out; ++i) { rm[i] = p->d_xout[0] + cplane * p->out_slot[outs[i]]; tl[i] = p->d_out[outs[i]]; }
        if ((rc = launch_conv(p, false, rm, tl, n_out, 0, 1, st))) return rc;
        for (int i = 0; i < n_out; ++i) {
            CU(cudaMemcpyAsync(p->h_out[outs[i]], rm[i], (size_t)p->pitch * sizeof(double), cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(p->h_bits[outs[i]], p->d_bits[outs[i]], (size_t)p->words_per_row * sizeof(uint32_t),
                               cudaMemcpyDeviceToHost, st));
        }
    }
    CU(cudaStreamSynchronize(st));
    for (int i = 0; i < n_out; ++i)
        if ((rc = pqb_panel_get_output(p, 0, outs[i], dst[i]->values, dst[i]->validity, n))) return rc;
    return PQB_OK;
}

static pqb_suite_params only(uint32_t ind) {
    pqb_suite_params sp;
    pqb_suite_params_default(&sp);
    sp.indicators = ind;
    return sp;
}

extern "C" int pqb_sma(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_SMA); sp.sma_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_SMA}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_ema(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_EMA); sp.ema_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_EMA}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_tema(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_TEMA); sp.tema_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_TEMA}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_trima(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_TRIMA); sp.trima_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_TRIMA}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_ma(pqb_engine *e, const pqb_col *real, int32_t tp, int32_t matype, pqb_out_col *out) {
    switch (matype) {                       // calc_ma overlap.rs:857-869
        case 1: return pqb_ema(e, real, tp, out);
        case 4: return pqb_tema(e, real, tp, out);
        case 5: return pqb_trima(e, real, tp, out);
        case 2: case 3: case 6: case 8:
            return fail(PQB_ERR_UNSUPPORTED, "matype %d (WMA/DEMA/KAMA/T3: defective in the reference, SURVEY 8a) is not built", matype);
        default: return pqb_sma(e, real, tp, out);
    }
}
extern "C" int pqb_bbands(pqb_engine *e, const pqb_col *real, int32_t tp, double up, double dn, pqb_out_col *u,
                          pqb_out_col *m, pqb_out_col *l) {
    pqb_suite_params sp = only(PQB_IND_BBANDS); sp.bbands_period = tp; sp.bbands_nbdevup = up; sp.bbands_nbdevdn = dn;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE};
    const int o[] = {PQB_OUT_BB_UPPER, PQB_OUT_BB_MIDDLE, PQB_OUT_BB_LOWER}; pqb_out_col *d[] = {u, m, l};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 3);
}
extern "C" int pqb_macd(pqb_engine *e, const pqb_col *real, int32_t fp, int32_t slp, int32_t sgp, pqb_out_col *m,
                        pqb_out_col *s, pqb_out_col *h) {
    pqb_suite_params sp = only(PQB_IND_MACD); sp.macd_fast = fp; sp.macd_slow = slp; sp.macd_signal = sgp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE};
    const int o[] = {PQB_OUT_MACD, PQB_OUT_MACD_SIGNAL, PQB_OUT_MACD_HIST}; pqb_out_col *d[] = {m, s, h};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 3);
}
extern "C" int pqb_rsi(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_RSI); sp.rsi_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_RSI}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_trange(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_TRANGE);
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_TRANGE};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_atr(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_ATR); sp.atr_period = tp;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_ATR};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_natr(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_NATR); sp.natr_period = tp;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_NATR};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_obv(pqb_engine *e, const pqb_col *cl, const pqb_col *v, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_OBV);
    const pqb_col *c[] = {cl, v}; const int f[] = {PQB_CLOSE, PQB_VOLUME}; const int o[] = {PQB_OUT_OBV};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 2, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_ad(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, const pqb_col *v, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_AD);
    const pqb_col *c[] = {h, l, cl, v}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE, PQB_VOLUME};
    const int o[] = {PQB_OUT_AD}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 4, NP_SHIFT, &sp, o, d, 1);
}
extern "C" int pqb_stoch(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t fk, int32_t sk,
                         int32_t sd, pqb_out_col *slowk, pqb_out_col *slowd) {
    pqb_suite_params sp = only(PQB_IND_KDJ); sp.kdj_fastk = fk; sp.kdj_slowk = sk; sp.kdj_slowd = sd;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE};
    const int o[] = {PQB_OUT_KDJ_K, PQB_OUT_KDJ_D}; pqb_out_col *d[] = {slowk, slowd};
    return run_single(e, c, f, 3, NP_SHIFT, &sp, o, d, 2);
}
extern "C" int pqb_kdj(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t fk, int32_t kp,
                       int32_t dp, pqb_out_col *k, pqb_out_col *dd, pqb_out_col *j) {
    pqb_suite_params sp = only(PQB_IND_KDJ); sp.kdj_fastk = fk; sp.kdj_slowk = kp; sp.kdj_slowd = dp;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE};
    const int o[] = {PQB_OUT_KDJ_K, PQB_OUT_KDJ_D, PQB_OUT_KDJ_J}; pqb_out_col *d[] = {k, dd, j};
    return run_single(e, c, f, 3, NP_SHIFT, &sp, o, d, 3);
}
extern "C" int pqb_willr(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_WILLR); sp.willr_period = tp;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_WILLR};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_midprice(pqb_engine *e, const pqb_col *h, const pqb_col *l, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_MIDPRICE); sp.midprice_period = tp;
    const pqb_col *c[] = {h, l}; const int f[] = {PQB_HIGH, PQB_LOW}; const int o[] = {PQB_OUT_MIDPRICE};
    pqb_out_col *d[] = {out};
    // nulls in `low` make the reference fail (overlap.rs:352-376); nulls in `high` alone would
    // need a per-field start: both are refused.
    return run_single(e, c, f, 2, NP_ERR, &sp, o, d, 1);
}

// ---- the remaining SURVEY.md 8a functions ----
extern "C" int pqb_midpoint(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_MIDPOINT); sp.midpoint_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_MIDPOINT}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_SHIFT, &sp, o, d, 1);    // (overlap.rs:180-278: a null bar emits null, the window skips it)
}
extern "C" int pqb_adosc(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, const pqb_col *v,
                         int32_t fp, int32_t slp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_ADOSC); sp.adosc_fast = fp; sp.adosc_slow = slp;
    const pqb_col *c[] = {h, l, cl, v}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE, PQB_VOLUME};
    const int o[] = {PQB_OUT_ADOSC}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 4, NP_SHIFT, &sp, o, d, 1);    // (calc_ad / calc_ema skip null bars)
}
extern "C" int pqb_mom(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_MOM); sp.mom_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_MOM}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_roc(pqb_engine *e, const pqb_col *real, int32_t tp, int32_t kind, pqb_out_col *out) {
    if (kind < 0 || kind > 3) return fail(PQB_ERR_INVALID, "pqb_roc: kind %d not in 0..3", kind);
    pqb_suite_params sp = only(PQB_IND_ROC); sp.roc_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_ROC + kind}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_cmo(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_CMO); sp.cmo_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_CMO}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_mfi(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, const pqb_col *v, int32_t tp,
                       pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_MFI); sp.mfi_period = tp;
    const pqb_col *c[] = {h, l, cl, v}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE, PQB_VOLUME};
    const int o[] = {PQB_OUT_MFI}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 4, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_cci(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_CCI); sp.cci_period = tp;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_CCI};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_ERR, &sp, o, d, 1);
}

extern "C" int pqb_trix(pqb_engine *e, const pqb_col *real, int32_t tp, pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_TRIX); sp.trix_period = tp;
    const pqb_col *c[] = {real}; const int f[] = {PQB_CLOSE}; const int o[] = {PQB_OUT_TRIX}; pqb_out_col *d[] = {out};
    return run_single(e, c, f, 1, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_ultosc(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t p1, int32_t p2, int32_t p3,
                          pqb_out_col *out) {
    pqb_suite_params sp = only(PQB_IND_ULTOSC); sp.ultosc_period1 = p1; sp.ultosc_period2 = p2; sp.ultosc_period3 = p3;
    const pqb_col *c[] = {h, l, cl}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE}; const int o[] = {PQB_OUT_ULTOSC};
    pqb_out_col *d[] = {out};
    return run_single(e, c, f, 3, NP_ERR, &sp, o, d, 1);
}
extern "C" int pqb_aroon(pqb_engine *e, const pqb_col *h, const pqb_col *l, int32_t tp, pqb_out_col *up, pqb_out_col *down) {
    pqb_suite_params sp = only(PQB_IND_AROON); sp.aroon_period = tp;
    const pqb_col *c[] = {h, l}; const int f[] = {PQB_HIGH, PQB_LOW};
    const int o[] = {PQB_OUT_AROON_UP, PQB_OUT_AROON_DOWN}; pqb_out_col *d[] = {up, down};
    return run_single(e, c, f, 2, NP_ERR, &sp, o, d, 2);
}
extern "C" int pqb_donchian(pqb_engine *e, const pqb_col *h, const pqb_col *l, int32_t tp, pqb_out_col *upper, pqb_out_col *lower) {
    pqb_suite_params sp = only(PQB_IND_DONCHIAN); sp.donchian_period = tp;
    const pqb_col *c[] = {h, l}; const int f[] = {PQB_HIGH, PQB_LOW};
    const int o[] = {PQB_OUT_DONCHIAN_UPPER, PQB_OUT_DONCHIAN_LOWER}; pqb_out_col *d[] = {upper, lower};
    return run_single(e, c, f, 2, NP_ERR, &sp, o, d, 2);
}
extern "C" int pqb_dm(pqb_engine *e, const pqb_col *h, const pqb_col *l, const pqb_col *cl, int32_t tp, pqb_out_col *plus_dm,
                      pqb_out_col *minus_dm, pqb_out_col *dx, pqb_out_col *minus_di, pqb_out_col *adx, pqb_out_col *adxr) {
    pqb_suite_params sp = only(PQB_IND_DM); sp.dm_period = tp;
    if (!h || !l) return fail(PQB_ERR_INVALID, "pqb_dm: high and low are required");
    const bool need_close = dx || minus_di || adx || adxr;
    if (need_close && !cl) return fail(PQB_ERR_INVALID, "pqb_dm: dx / minus_di / adx / adxr need close");
    // plus_dm / minus_dm alone (momentum.rs:362, :418) read high and low only: a stand-in close keeps the launch uniform
    const pqb_col *c[] = {h, l, cl ? cl : h}; const int f[] = {PQB_HIGH, PQB_LOW, PQB_CLOSE};
    pqb_out_col *all[] = {plus_dm, minus_dm, dx, minus_di, adx, adxr};
    int o[6]; pqb_out_col *d[6]; int n = 0;
    for (int k = 0; k < 6; ++k)
        if (all[k]) { o[n] = PQB_OUT_PLUS_DM + k; d[n] = all[k]; ++n; }
    if (n == 0) return fail(PQB_ERR_INVALID, "pqb_dm: no output requested");
    return run_single(e, c, f, 3, NP_ERR, &sp, o, d, n);
}

// ---------------------------------------------------------------------------------------
// multi-GPU driver: symbol shards, one host thread per shard, no collective
// ---------------------------------------------------------------------------------------
struct pqb_multi {
    struct Shard { int device = 0; int64_t lo = 0, hi = 0; pqb_engine *e = nullptr; pqb_panel *p = nullptr; };
    std::vector<Shard> shards;
    int64_t n_symbols = 0, n_bars = 0;
};

extern "C" void pqb_multi_destroy(pqb_multi *m) {
    if (!m) return;
    for (auto &s : m->shards) {
        if (s.p) pqb_panel_destroy(s.p);
        if (s.e) pqb_engine_destroy(s.e);
    }
    delete m;
}

extern "C" int pqb_multi_create(const int *devices, int n_devices, int64_t n_symbols, int64_t n_bars,
                                uint32_t fields_mask, uint64_t outputs_mask, pqb_multi **out) {
    if (!devices || n_devices <= 0 || !out) return fail(PQB_ERR_INVALID, "pqb_multi_create: bad argument");
    *out = nullptr;
    if (n_symbols <= 0 || n_bars <= 0) return fail(PQB_ERR_INVALID, "pqb_multi_create: bad shape");
    pqb_multi *m = new pqb_multi();
    m->n_symbols = n_symbols;
    m->n_bars = n_bars;
    // contiguous ranges of whole 32-symbol blocks, balanced to one block (polars_quant_b200/shard.py)
    const int64_t n_blocks = (n_symbols + SYM - 1) / SYM;
    const int64_t base = n_blocks / n_devices, extra = n_blocks % n_devices;
    for (int r = 0; r < n_devices; ++r) {
        const int64_t b_lo = r * base + std::min<int64_t>(r, extra), b_hi = b_lo + base + (r < extra ? 1 : 0);
        pqb_multi::Shard s;
        s.device = devices[r];
        s.lo = std::min(b_lo * SYM, n_symbols);
        s.hi = std::min(b_hi * SYM, n_symbols);
        if (s.hi > s.lo) {
            int rc = pqb_engine_create(s.device, &s.e);
            if (!rc) rc = pqb_panel_create(s.e, s.hi - s.lo, n_bars, fields_mask, outputs_mask, 1, &s.p);
            if (rc) { m->shards.push_back(s); pqb_multi_destroy(m); return rc; }
        }
        m->shards.push_back(s);
    }
    *out = m;
    return PQB_OK;
}

extern "C" int pqb_multi_shard_count(const pqb_multi *m) { return m ? (int)m->shards.size() : 0; }

extern "C" int pqb_multi_shard(const pqb_multi *m, int i, int *device, int64_t *lo, int64_t *hi, pqb_panel **panel) {
    if (!m || i < 0 || i >= (int)m->shards.size()) return fail(PQB_ERR_INVALID, "pqb_multi_shard: bad index");
    const auto &s = m->shards[(size_t)i];
    if (device) *device = s.device;
    if (lo) *lo = s.lo;
    if (hi) *hi = s.hi;
    if (panel) *panel = s.p;
    return PQB_OK;
}

static const pqb_multi::Shard *shard_of(const pqb_multi *m, int64_t symbol) {
    for (const auto &s : m->shards)
        if (symbol >= s.lo && symbol < s.hi) return &s;
    return nullptr;
}

extern "C" int pqb_multi_set_column(pqb_multi *m, int64_t symbol, int field, const double *values,
                                    const uint8_t *validity, int64_t offset, int64_t len) {
    const pqb_multi::Shard *s = m ? shard_of(m, symbol) : nullptr;
    if (!s) return fail(PQB_ERR_INVALID, "pqb_multi_set_column: symbol %lld out of range", (long long)symbol);
    return pqb_panel_set_column(s->p, symbol - s->lo, field, values, validity, offset, len);
}

extern "C" int pqb_multi_get_output(pqb_multi *m, int64_t symbol, int output, double *values, uint8_t *validity,
                                    int64_t len) {
    const pqb_multi::Shard *s = m ? shard_of(m, symbol) : nullptr;
    if (!s) return fail(PQB_ERR_INVALID, "pqb_multi_get_output: symbol %lld out of range", (long long)symbol);
    return pqb_panel_get_output(s->p, symbol - s->lo, output, values, validity, len);
}

extern "C" int pqb_multi_run_host(pqb_multi *m, const pqb_suite_params *params) {
    if (!m || !params) return fail(PQB_ERR_INVALID, "pqb_multi_run_host: NULL argument");
    const size_t n = m->shards.size();
    std::vector<int> rcs(n, PQB_OK);
    std::vector<std::string> errs(n);
    std::vector<std::thread> th;
    for (size_t i = 0; i < n; ++i) {
        if (!m->shards[i].p) continue;
        th.emplace_back([&, i] {
            rcs[i] = pqb_suite_run_host(m->shards[i].p, params, 0);
            if (rcs[i]) errs[i] = g_err;                  // the error text is thread-local: carry it over
        });
    }
    for (auto &t : th) t.join();
    for (size_t i = 0; i < n; ++i)
        if (rcs[i]) return fail(rcs[i], "shard %zu (device %d, symbols [%lld, %lld)): %s", i, m->shards[i].device,
                                (long long)m->shards[i].lo, (long long)m->shards[i].hi, errs[i].c_str());
    return PQB_OK;
}

#include "columns_host.inc"
#include "candles_host.inc"
#include "split_host.inc"
#include "longrows_host.inc"
#include "windows_host.inc"
#include "shims_host.inc"
#include "signals_host.inc"
#include "info_host.inc"
#include "live_host.inc"
