// candles.cuh -- fused candle kernel for sm_100a: the reference's 61 candlestick patterns
// (src/talib/pattern.rs:9-2065, Int32 outputs in {-100, 0, 100}), the four price transforms
// (src/talib/price.rs:10-91) and BOP (src/talib/momentum.rs:113-135) from open / high / low / close
// in ONE pass (SURVEY.md 8f.1).
//
// The reference runs 66 separate plugin calls per symbol, each re-reading the four columns and each
// re-deriving the same per-bar quantities (body, shadows, long / short / doji tests) for up to five
// bars.  Here a bar's shape is classified ONCE into a 16-bit flag word; every pattern is then a
// boolean combination of the flag words of bars t .. t-4 plus a few cross-bar comparisons of raw
// prices, so the whole family costs ~35 FP64 operations per bar instead of ~600.
//
// Layout: row-major [symbol][pitch] planes -- the Arrow-shaped layout of the ABI -- because this is a
// pure stencil: a warp takes 32 consecutive bars of one symbol (256 B per input plane, 128 B per Int32
// output plane, whole cache lines either way), a CTA 256 consecutive bars (+4 halo bars) staged in
// shared memory.  HBM-bound: 32 B in + 4 B x patterns + 8 B x prices per symbol-bar (316 B with
// everything enabled), every output written exactly once with streaming stores.
// Arithmetic is f64 in the reference's expression order (-fmad=false), comparisons only: results
// are bit-exact.  Nulls: patterns and BOP refuse them on the host like the reference's cont_slice()?;
// the price transforms propagate them (validity word = AND of the inputs' words, one ballot per warp).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pqb {

// pattern ids: the reference's (alphabetical) order of definition in pattern.rs
#define PQB_PATTERN_LIST(X)                                                                                  \
    X(cdl2crows) X(cdl3blackcrows) X(cdl3inside) X(cdl3linestrike) X(cdl3outside) X(cdl3starsinsouth)        \
    X(cdl3whitesoldiers) X(cdlabandonedbaby) X(cdladvanceblock) X(cdlbelthold) X(cdlbreakaway)               \
    X(cdlclosingmarubozu) X(cdlconcealbabyswall) X(cdlcounterattack) X(cdldarkcloudcover) X(cdldoji)         \
    X(cdldojistar) X(cdldragonflydoji) X(cdlengulfing) X(cdleveningdojistar) X(cdleveningstar)               \
    X(cdlgapsidesidewhite) X(cdlgravestonedoji) X(cdlhammer) X(cdlhangingman) X(cdlharami) X(cdlharamicross) \
    X(cdlhighwave) X(cdlhikkake) X(cdlhikkakemod) X(cdlhomingpigeon) X(cdlidentical3crows) X(cdlinneck)      \
    X(cdlinvertedhammer) X(cdlkicking) X(cdlkickingbylength) X(cdlladderbottom) X(cdllongleggeddoji)         \
    X(cdllongline) X(cdlmarubozu) X(cdlmatchinglow) X(cdlmathold) X(cdlmorningdojistar) X(cdlmorningstar)    \
    X(cdlonneck) X(cdlpiercing) X(cdlrickshawman) X(cdlrisefall3methods) X(cdlseparatinglines)               \
    X(cdlshootingstar) X(cdlshortline) X(cdlspinningtop) X(cdlstalledpattern) X(cdlsticksandwich)            \
    X(cdltakuri) X(cdltasukigap) X(cdlthrusting) X(cdltristar) X(cdlunique3river) X(cdlupsidegap2crows)      \
    X(cdlxsidegap3methods)

enum PatternId {
#define X(n) P_##n,
    PQB_PATTERN_LIST(X)
#undef X
    N_PATTERNS
};
static_assert(N_PATTERNS == 61, "pattern.rs defines 61 functions");

constexpr int N_PRICES = 5;          // avgprice, medprice, typprice, wclprice, bop
constexpr int CANDLE_TILE = 256;     // bars per CTA
constexpr int CANDLE_HALO = 4;       // deepest lookback (breakaway, ladderbottom, mathold, risefall3methods)

// the six functions that read a `penetration` literal (pattern.rs `inputs.get(4) ... unwrap_or(0.3)`)
enum { PEN_DARKCLOUDCOVER, PEN_EVENINGDOJISTAR, PEN_EVENINGSTAR, PEN_MORNINGDOJISTAR, PEN_MORNINGSTAR, PEN_PIERCING, N_PEN };

struct CandleArgs {
    const double *in[4];             // open, high, low, close: row-major [n_symbols][pitch]
    const uint32_t *vin[4];          // input validity words [n_symbols][words_per_row] or nullptr (all valid)
    int32_t *pat[N_PATTERNS];        // Int32 planes [n_symbols][pitch] or nullptr
    double *price[N_PRICES];         // f64 planes or nullptr
    uint32_t *vprice[N_PRICES];      // validity words of the price planes or nullptr
    double pen[N_PEN];
    size_t pat_stride;               // ALL specialisation: pattern k's plane = pat[0] + k * pat_stride (one allocation)
    int n_symbols, n_bars, pitch, words_per_row;
    int symbol0;                     // first symbol of this launch (chunked host pipeline)
};

// per-bar shape flags (pattern.rs:2068-2143 helper predicates, each evaluated once per bar)
enum : unsigned {
    CF_BULL = 1u << 0,    // c > o
    CF_BEAR = 1u << 1,    // c < o
    CF_LONG = 1u << 2,    // |o-c| > 0.05 * (o+c) * 0.5
    CF_SHORT = 1u << 3,   // |o-c| < 0.1 * (o+c) * 0.5
    CF_DOJI = 1u << 4,    // |o-c| <= 0.005 * (o+c) * 0.5
    CF_LUS = 1u << 5,     // upper shadow > 2 body
    CF_LDS = 1u << 6,     // lower shadow > 2 body
    CF_SUS = 1u << 7,     // upper shadow < 0.5 body
    CF_SDS = 1u << 8,     // lower shadow < 0.5 body
    CF_VSUS = 1u << 9,    // upper shadow < 0.1 body
    CF_VSDS = 1u << 10,   // lower shadow < 0.1 body
    CF_VLDS = 1u << 11,   // lower shadow > 3 body
    CF_USGB = 1u << 12,   // upper shadow > body   (spinningtop)
    CF_LSGB = 1u << 13,   // lower shadow > body
};

__device__ __forceinline__ unsigned classify(double o, double h, double l, double c) {
    const double body = fabs(o - c);
    const double sum = o + c;
    const double us = h - fmax(o, c);          // Rust f64::max / min: a NaN operand is ignored, like fmax / fmin
    const double ls = fmin(o, c) - l;
    unsigned f = 0;
    f |= (c > o) ? CF_BULL : 0u;
    f |= (c < o) ? CF_BEAR : 0u;
    f |= (body > 0.05 * sum * 0.5) ? CF_LONG : 0u;
    f |= (body < 0.1 * sum * 0.5) ? CF_SHORT : 0u;
    f |= (body <= 0.005 * sum * 0.5) ? CF_DOJI : 0u;
    const double b2 = 2.0 * body, bh = 0.5 * body, bt = 0.1 * body;
    f |= (us > b2) ? CF_LUS : 0u;
    f |= (ls > b2) ? CF_LDS : 0u;
    f |= (us < bh) ? CF_SUS : 0u;
    f |= (ls < bh) ? CF_SDS : 0u;
    f |= (us < bt) ? CF_VSUS : 0u;
    f |= (ls < bt) ? CF_VSDS : 0u;
    f |= (ls > 3.0 * body) ? CF_VLDS : 0u;
    f |= (us > body) ? CF_USGB : 0u;
    f |= (ls > body) ? CF_LSGB : 0u;
    return f;
}

__device__ __forceinline__ void st_i32(int32_t *p, int v) { __stcs(p, v); }

// grid = (ceil(n_bars / CANDLE_TILE), symbols of this launch), CANDLE_TILE threads.
// ALL: every pattern enabled and the 61 planes are one allocation (no mask tests, one base pointer).
template <bool ALL>
__global__ void __launch_bounds__(CANDLE_TILE, 3) candle_kernel(const __grid_constant__ CandleArgs A, const uint64_t pmask) {
    __shared__ double so[CANDLE_TILE + CANDLE_HALO], sh[CANDLE_TILE + CANDLE_HALO], sl[CANDLE_TILE + CANDLE_HALO],
        sc[CANDLE_TILE + CANDLE_HALO];
    __shared__ unsigned short sf[CANDLE_TILE + CANDLE_HALO];
    const int tid = threadIdx.x;
    const int s = A.symbol0 + blockIdx.y;
    const int t0 = blockIdx.x * CANDLE_TILE;
    const int i = t0 + tid;                                  // this thread's bar
    const size_t row = (size_t)s * A.pitch;
    const bool live = i < A.n_bars;

    // ---- stage the tile (+ halo) and classify every bar once
    double o0 = 0.0, h0 = 0.0, l0 = 0.0, c0 = 0.0;
    if (live) {
        o0 = __ldg(A.in[0] + row + i);
        h0 = __ldg(A.in[1] + row + i);
        l0 = __ldg(A.in[2] + row + i);
        c0 = __ldg(A.in[3] + row + i);
    }
    const unsigned f0 = classify(o0, h0, l0, c0);
    so[tid + CANDLE_HALO] = o0; sh[tid + CANDLE_HALO] = h0; sl[tid + CANDLE_HALO] = l0; sc[tid + CANDLE_HALO] = c0;
    sf[tid + CANDLE_HALO] = (unsigned short)f0;
    if (tid < CANDLE_HALO) {
        const int j = t0 - CANDLE_HALO + tid;
        double o = 0.0, h = 0.0, l = 0.0, c = 0.0;
        if (j >= 0) {
            o = __ldg(A.in[0] + row + j);
            h = __ldg(A.in[1] + row + j);
            l = __ldg(A.in[2] + row + j);
            c = __ldg(A.in[3] + row + j);
        }
        so[tid] = o; sh[tid] = h; sl[tid] = l; sc[tid] = c;
        sf[tid] = (unsigned short)classify(o, h, l, c);
    }
    __syncthreads();

    // ---- price transforms + BOP (null-propagating: validity = AND of the inputs' words; one word per warp)
    {
        const int w = i >> 5;                                // validity word of this warp's 32 bars (t0 is a multiple of 32)
        unsigned vo = 0xffffffffu, vh = vo, vl = vo, vc = vo;
        if (live) {
            const size_t wi = (size_t)s * A.words_per_row + w;
            if (A.vin[0]) vo = A.vin[0][wi];
            if (A.vin[1]) vh = A.vin[1][wi];
            if (A.vin[2]) vl = A.vin[2][wi];
            if (A.vin[3]) vc = A.vin[3][wi];
        }
        const unsigned bit = 1u << (tid & 31);
        const bool ko = vo & bit, kh = vh & bit, kl = vl & bit, kc = vc & bit;
        const double nn = __longlong_as_double(0x7ff8000000000000LL);
        auto emit = [&](int k, double v, bool ok) {
            if (!A.price[k]) return;
            ok = ok && live;
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (live) {
                __stcs(A.price[k] + row + i, ok ? v : nn);
                if ((tid & 31) == 0 && A.vprice[k]) A.vprice[k][(size_t)s * A.words_per_row + w] = m;
            }
        };
#include "candle_prices.inc"
    }
    if (!ALL && pmask == 0) return;

    // ---- the window: k bars back = index tid + HALO - k
    const int q = tid + CANDLE_HALO;
    const double o1 = so[q - 1], h1 = sh[q - 1], l1 = sl[q - 1], c1 = sc[q - 1];
    const double o2 = so[q - 2], h2 = sh[q - 2], l2 = sl[q - 2], c2 = sc[q - 2];
    const double o3 = so[q - 3], h3 = sh[q - 3], l3 = sl[q - 3], c3 = sc[q - 3];
    const double o4 = so[q - 4], h4 = sh[q - 4], l4 = sl[q - 4], c4 = sc[q - 4];
    const unsigned f1 = sf[q - 1], f2 = sf[q - 2], f3 = sf[q - 3], f4 = sf[q - 4];
    const size_t at = row + i;
    int32_t *const pbase = A.pat[0] + at;
    const size_t pstride = A.pat_stride;
#define HAS(f, m) (((f) & (m)) == (m))
#define NEAR(a, b) (fabs((a) - (b)) < near_t)
#define EQUAL(a, b) (fabs((a) - (b)) < equal_t)
    // `up` -> +100, else `dn` -> -100, else 0.  (A warp-voted early-out on the flag preconditions was measured:
    // on random-walk data almost every 32-bar warp has a lane that passes, and the votes cost more than they save.)
#define EMIT(id, up, dn)                                                                   \
    if (ALL || (pmask >> (id) & 1)) {                                                      \
        if (live) st_i32(ALL ? pbase + (size_t)(id) * pstride : A.pat[id] + at, (up) ? 100 : ((dn) ? -100 : 0)); \
    }
#include "candle_patterns.inc"
#undef EMIT
#undef HAS
#undef NEAR
#undef EQUAL
    (void)pstride; (void)pbase;
}

// ---- live candle panels (candles_live_host.inc): append bars to a candle panel ------------------------------------
// A pushed bar's row needs the 4 bars before it and nothing after it, so a live panel keeps the latest CANDLE_HALO bars of
// each field (the tail) and each thread walks one symbol through the tail and the pushed bars.  Bar-major rows
// [bar][n_symbols]: a warp's 32 consecutive symbols load one 256-byte line per field and bar and store 128 bytes per
// Int32 row; price validity is the warp's ballot word, 4 bytes of the bar's LSB-first row bitmap.
constexpr int CANDLE_LIVE_THREADS = 32;   // one warp per CTA: the few warps of a panel spread evenly over the SMs

struct CandleLiveArgs {
    const double *rows[4];           // pushed bars of open, high, low, close: [k][n_symbols], or nullptr (unread field: 0.0)
    const uint32_t *vrows[4];        // their validity words [k][row_words], or nullptr (all valid)
    const double *tail_in;           // bars T-4 .. T-1: [field][CANDLE_HALO][n_symbols] (0.0 before bar 0)
    double *tail_out;                // the same after the push, or nullptr (a preview)
    int32_t *pat[N_PATTERNS];        // Int32 rows [k][n_symbols] or nullptr
    double *price[N_PRICES];         // f64 rows [k][n_symbols] or nullptr
    uint32_t *vprice[N_PRICES];      // their validity words [k][row_words]
    double pen[N_PEN];
    size_t pat_stride;               // ALL: pattern k's rows = pat[0] + k * pat_stride
    int n_symbols, k, row_words;
    int t_base;                      // absolute index of the first pushed bar (the bars before the push, T)
};

// grid = ceil(n_symbols / CANDLE_LIVE_THREADS).  Every bar is classified once; the pattern block is candle_kernel's text,
// evaluated at the absolute bar index, so the lookback guards and the zeros before bar 0 are the full panel's.
template <bool ALL>
__global__ void __launch_bounds__(CANDLE_LIVE_THREADS) candle_live_kernel(const __grid_constant__ CandleLiveArgs A, const uint64_t pmask) {
    const int s = blockIdx.x * CANDLE_LIVE_THREADS + threadIdx.x;
    const bool live = s < A.n_symbols;
    const size_t n = (size_t)A.n_symbols;
    const int w = s >> 5;                                    // this warp's validity word in a row
    auto tail = [&](int f, int j) { return live ? __ldg(A.tail_in + ((size_t)f * CANDLE_HALO + j) * n + s) : 0.0; };
    double o4 = tail(0, 0), h4 = tail(1, 0), l4 = tail(2, 0), c4 = tail(3, 0);
    double o3 = tail(0, 1), h3 = tail(1, 1), l3 = tail(2, 1), c3 = tail(3, 1);
    double o2 = tail(0, 2), h2 = tail(1, 2), l2 = tail(2, 2), c2 = tail(3, 2);
    double o1 = tail(0, 3), h1 = tail(1, 3), l1 = tail(2, 3), c1 = tail(3, 3);
    unsigned f4 = classify(o4, h4, l4, c4), f3 = classify(o3, h3, l3, c3), f2 = classify(o2, h2, l2, c2),
             f1 = classify(o1, h1, l1, c1);
    const double nn = __longlong_as_double(0x7ff8000000000000LL);
    for (int t = 0; t < A.k; ++t) {
        const int i = A.t_base + t;                          // absolute bar index
        const size_t at = (size_t)t * n + s;
        double o0 = 0.0, h0 = 0.0, l0 = 0.0, c0 = 0.0;
        if (live) {
            if (A.rows[0]) o0 = __ldg(A.rows[0] + at);
            if (A.rows[1]) h0 = __ldg(A.rows[1] + at);
            if (A.rows[2]) l0 = __ldg(A.rows[2] + at);
            if (A.rows[3]) c0 = __ldg(A.rows[3] + at);
        }
        const unsigned f0 = classify(o0, h0, l0, c0);
        {
            unsigned vo = 0xffffffffu, vh = vo, vl = vo, vc = vo;
            const size_t wi = (size_t)t * A.row_words + w;
            if (live) {
                if (A.vrows[0]) vo = __ldg(A.vrows[0] + wi);
                if (A.vrows[1]) vh = __ldg(A.vrows[1] + wi);
                if (A.vrows[2]) vl = __ldg(A.vrows[2] + wi);
                if (A.vrows[3]) vc = __ldg(A.vrows[3] + wi);
            }
            const unsigned bit = 1u << (threadIdx.x & 31);
            const bool ko = vo & bit, kh = vh & bit, kl = vl & bit, kc = vc & bit;
            auto emit = [&](int k, double v, bool ok) {
                if (!A.price[k]) return;
                ok = ok && live;
                const unsigned m = __ballot_sync(0xffffffffu, ok);
                if (live) {
                    A.price[k][at] = ok ? v : nn;
                    if ((threadIdx.x & 31) == 0 && A.vprice[k]) A.vprice[k][wi] = m;
                }
            };
#include "candle_prices.inc"
        }
        if (ALL || pmask) {
            int32_t *const pbase = A.pat[0] + at;
            const size_t pstride = A.pat_stride;
#define HAS(f, m) (((f) & (m)) == (m))
#define NEAR(a, b) (fabs((a) - (b)) < near_t)
#define EQUAL(a, b) (fabs((a) - (b)) < equal_t)
#define EMIT(id, up, dn)                                                                                  \
    if (ALL || (pmask >> (id) & 1)) {                                                                     \
        if (live) *(ALL ? pbase + (size_t)(id) * pstride : A.pat[id] + at) = (up) ? 100 : ((dn) ? -100 : 0); \
    }
#include "candle_patterns.inc"
#undef EMIT
#undef HAS
#undef NEAR
#undef EQUAL
            (void)pstride; (void)pbase;
        }
        o4 = o3; h4 = h3; l4 = l3; c4 = c3; f4 = f3;
        o3 = o2; h3 = h2; l3 = l2; c3 = c2; f3 = f2;
        o2 = o1; h2 = h1; l2 = l1; c2 = c1; f2 = f1;
        o1 = o0; h1 = h0; l1 = l0; c1 = c0; f1 = f0;
    }
    if (A.tail_out && live) {
        auto put = [&](int j, double o, double h, double l, double c) {
            A.tail_out[((size_t)0 * CANDLE_HALO + j) * n + s] = o;
            A.tail_out[((size_t)1 * CANDLE_HALO + j) * n + s] = h;
            A.tail_out[((size_t)2 * CANDLE_HALO + j) * n + s] = l;
            A.tail_out[((size_t)3 * CANDLE_HALO + j) * n + s] = c;
        };
        put(0, o4, h4, l4, c4);
        put(1, o3, h3, l3, c3);
        put(2, o2, h2, l2, c2);
        put(3, o1, h1, l1, c1);
    }
}

// synthetic candle panel for the bench (device-side, counter-based): a random walk of opens with bodies and
// shadows of mixed sizes on a 0.01 price grid, so that patterns do fire
__global__ void candle_synth_kernel(double *o, double *h, double *l, double *c, int n_symbols, int n_bars, int pitch,
                                    unsigned long long seed) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_symbols) return;
    unsigned long long x = seed * 0x9E3779B97F4A7C15ull + (unsigned long long)s * 0xD1B54A32D192ED03ull + 1;
    auto rnd = [&]() {                     // splitmix64 -> [0, 1)
        x += 0x9E3779B97F4A7C15ull;
        unsigned long long z = x;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        return (double)(z >> 11) * (1.0 / 9007199254740992.0);
    };
    double prev = 50.0 + (s % 97);
    for (int t = 0; t < n_bars; ++t) {
        const double g = rnd();
        double op = prev * (1.0 + (g < 0.15 ? 0.02 : (g < 0.3 ? -0.02 : 0.0)));
        const double k = rnd();
        const double body = op * (k < 0.2 ? 0.0 : (k < 0.5 ? 0.01 * rnd() : 0.03 + 0.09 * rnd()));
        double cl = op + (rnd() < 0.5 ? -body : body);
        const double u = rnd(), d = rnd();
        double hi = fmax(op, cl) + op * (u < 0.4 ? 0.0 : (u < 0.7 ? 0.004 : 0.06 * rnd()));
        double lo = fmin(op, cl) - op * (d < 0.4 ? 0.0 : (d < 0.7 ? 0.004 : 0.06 * rnd()));
        op = rint(op * 100.0) / 100.0; cl = rint(cl * 100.0) / 100.0;
        hi = fmax(rint(hi * 100.0) / 100.0, fmax(op, cl));
        lo = fmax(0.01, fmin(rint(lo * 100.0) / 100.0, fmin(op, cl)));
        const size_t at = (size_t)s * pitch + t;
        o[at] = op; h[at] = hi; l[at] = lo; c[at] = cl;
        prev = fmax(5.0, cl);
    }
}

}  // namespace pqb
