// longrows.cuh -- few symbols, very long rows (BASELINE config 3: 500 symbols x 1,000,000 minute bars): K exponential
// moving averages + MACD in ONE pass over close, parallel along TIME.
//
// The fused suite kernel walks a symbol's time axis serially; 500 symbols are 16 symbol blocks for 444 CTA slots.  The
// EMA family (calc_ema overlap.rs:660-730, macd momentum.rs:250-283) is a chain of affine maps
//     y_t = (1 - alpha) * y_{t-1} + alpha * x_t          (the reference evaluates it as alpha.mul_add(x - y, y))
// so a row is cut into tiles of L bars and the state is carried across tiles by composing the tiles' maps
// (north_star: "affine-composition scans for the EMA, MACD and Wilder-RSI recurrences"):
//   seed   (lr_seed_kernel)   per chain: the reference's seed = (x_0 + ... + x_{p-1}) / p, summed left to right like
//                             the reference, emitted at bar p-1
//   local  (lr_local_kernel)  per (tile, symbol block): the tile's end state from a ZERO start, B_k (the tile's affine
//                             map is y -> A y + B_k with the same A = (1 - alpha)^L for every tile); for the MACD signal
//                             line, an EMA of dif = fast - slow, the local part from the local fast / slow states
//   carry  (lr_carry_kernel)  per symbol: y_k = A y_{k-1} + B_k over the tiles (977 steps of one fma at config 3); the
//                             signal's carry adds Cf * fast_{k-1} - Cs * slow_{k-1}, the closed-form contribution of the
//                             fast / slow start states to the tile's dif values
//   final  (lr_final_kernel)  per (tile, symbol block): starts from the carried state and walks the tile's bars in the
//                             REFERENCE'S OWN operation order (fma(alpha, x - y, y), dif = f - s, hist = dif - signal),
//                             writing every output once
// Tile 0 (and the tile that holds a chain's seed bar) is the reference's computation itself; later tiles differ from the
// serial walk only through the rounding of the carried start state (a few ulp of the state): EMA lines within rel 1e-10 /
// abs 1e-12, MACD lines within that + 4 ulp of the row's largest |close| -- tolerance-exact, not bit-exact, like the
// time-split panels of split_host.inc, but with no warm-up recomputation: 72 B of traffic per symbol-bar (close read
// twice) against 64 B algorithmic, whatever the period.
// Layout: the tiled planes of suite_kernel.cuh ([symbol block][bar][32 symbols]); lane = symbol, one warp = one
// (tile, block) unit reading / writing 256 contiguous bytes per plane per bar.
#pragma once
#include "suite_kernel.cuh"

namespace pqb {

constexpr int LR_MAX_CH = 8;      // distinct EMA chains of one launch (the MACD fast / slow EMAs share a chain with an equal period)
constexpr int LR_MAX_EMA = 7;     // EMA output planes
constexpr int LR_BATCH = 16;      // bars loaded ahead per lane

struct LongArgs {
    const double *x;                   // close, tiled
    double *chain_out[LR_MAX_CH];      // tiled output plane of chain c's EMA, or nullptr (a chain that only feeds the MACD)
    double *macd_out[3];               // macd, macd_signal, macd_hist
    int macd;                          // MACD on: chains 0 and 1 are its fast and slow EMA (fixed slots: registers, no indexing)
    int n_ch;                          // distinct chains
    int p[LR_MAX_CH];                  // period
    double alpha[LR_MAX_CH];           // 2 / (p + 1)                     overlap.rs:669
    double A[LR_MAX_CH];               // (1 - alpha)^L
    int macd_f, macd_s, macd_g;
    double alpha_g, A_g, Cf, Cs;       // signal chain: alpha, (1 - alpha_g)^L, start-state couplings (see lr_carry_kernel)
    double *seed;                      // [n_ch][n_blocks * 32]
    double *agg;                       // [n_tiles][n_ch + 1][n_blocks * 32]: the tiles' local end states B_k
    double *carry;                     // same shape: the carried end states y_k
    int n_symbols, n_bars, n_blocks, bars_padded, L, n_tiles;
    int max_p;                         // the longest period: tiles starting at or after it are past every seed bar
};

__device__ __forceinline__ double ld_stream(const double *p) { return __ldcs(p); }

// ---- seed: one warp per (symbol block, chain) -------------------------------------------------------------------------
__global__ void __launch_bounds__(32) lr_seed_kernel(const __grid_constant__ LongArgs A) {
    const int lane = threadIdx.x, b = blockIdx.x, c = blockIdx.y;
    const int p = A.p[c];
    const double *x = A.x + (size_t)b * A.bars_padded * SYM + lane;
    double sum = 0.0;
    if (p <= A.n_bars)
        for (int t = 0; t < p; ++t) sum += x[(size_t)t * SYM];          // left to right, like the reference (:689-693)
    A.seed[(size_t)c * A.n_blocks * SYM + b * SYM + lane] = sum / (double)p;       // :696
}

// the state of the MACD lines in tile 0: the reference's own count-based logic (Ema::step of suite_kernel.cuh)
struct MacdHead {
    Ema mf, ms, mg;
    __device__ __forceinline__ void init() { mf.init(); ms.init(); mg.init(); }
    __device__ __forceinline__ void step(const LongArgs &A, double c, int t, double &dif, double &sig, bool &okd, bool &okg) {
        const bool okf = mf.step<false>(c, t, A.macd_f, A.alpha[0]);
        const bool oks = ms.step<false>(c, t, A.macd_s, A.alpha[1]);
        okd = okf && oks;
        dif = mf.y - ms.y;                                               // momentum.rs:264
        okg = mg.step<false>(okd ? dif : 0.0, t, A.macd_g, A.alpha_g);   // unwrap_or(0.0) :269
        sig = mg.y;
    }
};

// ---- local: the end state of every chain over one tile from a zero start ---------------------------------------------------
// Interior tiles (every chain past its seed, a whole tile) take a straight-line path with a compile-time chain count:
// y = fma(1 - alpha, y, alpha * x) -- one dependent operation per bar and chain; its rounding differs from the
// reference's fma(alpha, x - y, y) only in the last place of a state that is re-rounded by the carry anyway.  Tile 0, the
// tiles holding a seed bar and the ragged last tile take the general path.
template <int NCH, bool MACD>
__device__ __forceinline__ void lr_local_fast(const LongArgs &A, const double *x, double *out, size_t lanes) {
    double y[NCH], a1[NCH], al[NCH], g = 0.0;
#pragma unroll
    for (int c = 0; c < NCH; ++c) { y[c] = 0.0; al[c] = A.alpha[c]; a1[c] = 1.0 - A.alpha[c]; }
    const double ag = A.alpha_g, ag1 = 1.0 - A.alpha_g;
    for (int tb = 0; tb < A.L; tb += LR_BATCH) {
        double xv[LR_BATCH];
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) xv[i] = ld_stream(x + (size_t)(tb + i) * SYM);
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) {
#pragma unroll
            for (int c = 0; c < NCH; ++c) y[c] = fma(a1[c], y[c], al[c] * xv[i]);
            if (MACD) g = fma(ag1, g, ag * (y[0] - y[1]));
        }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) out[(size_t)c * lanes] = y[c];
    out[(size_t)NCH * lanes] = g;
}

template <bool MACD>
__global__ void __launch_bounds__(128) lr_local_kernel(const __grid_constant__ LongArgs A) {
    const int lane = threadIdx.x & 31;
    const long long unit = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (unit >= (long long)A.n_tiles * A.n_blocks) return;
    const int tt = (int)(unit / A.n_blocks), b = (int)(unit % A.n_blocks);      // time-major: neighbouring warps share a tile index
    const int t0 = tt * A.L, t1 = min(t0 + A.L, A.n_bars);
    const double *x = A.x + ((size_t)b * A.bars_padded + t0) * SYM + lane;
    const size_t lanes = (size_t)A.n_blocks * SYM;
    double *out = A.agg + (size_t)tt * (A.n_ch + 1) * lanes + b * SYM + lane;
    if (tt > 0 && t0 >= A.max_p && t1 - t0 == A.L) {           // interior tile: every chain runs over the whole tile
        switch (A.n_ch) {
            case 1: lr_local_fast<1, MACD>(A, x, out, lanes); return;
            case 2: lr_local_fast<2, MACD>(A, x, out, lanes); return;
            case 3: lr_local_fast<3, MACD>(A, x, out, lanes); return;
            case 4: lr_local_fast<4, MACD>(A, x, out, lanes); return;
            case 5: lr_local_fast<5, MACD>(A, x, out, lanes); return;
            case 6: lr_local_fast<6, MACD>(A, x, out, lanes); return;
            default: break;
        }
    }
    double y[LR_MAX_CH];
    int from[LR_MAX_CH];                   // first bar of the tile at which chain c runs its recurrence
#pragma unroll
    for (int c = 0; c < LR_MAX_CH; ++c) {
        y[c] = 0.0;
        from[c] = t0;
        if (c < A.n_ch) {
            const int ts = A.p[c] - 1;     // the seed bar
            if (ts >= t1) from[c] = t1;                                   // tile entirely before the seed: nothing
            else if (ts >= t0) { from[c] = ts + 1; y[c] = A.seed[(size_t)c * lanes + b * SYM + lane]; }
        }
    }
    MacdHead head;
    double g = 0.0;
    if (MACD && tt == 0) head.init();
    for (int tb = t0; tb < t1; tb += LR_BATCH) {
        double xv[LR_BATCH];
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) xv[i] = (tb + i < t1) ? ld_stream(x + (size_t)(tb - t0 + i) * SYM) : 0.0;
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) {
            const int t = tb + i;
            if (t >= t1) break;
#pragma unroll
            for (int c = 0; c < LR_MAX_CH; ++c)
                if (c < A.n_ch && t >= from[c]) y[c] = fma(A.alpha[c], xv[i] - y[c], y[c]);
            if (MACD) {
                if (tt == 0) {
                    double dif, sig; bool okd, okg;
                    head.step(A, xv[i], t, dif, sig, okd, okg);
                    g = sig;
                } else {
                    const double dif = y[0] - y[1];
                    g = fma(A.alpha_g, dif - g, g);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < LR_MAX_CH; ++c)
        if (c < A.n_ch) out[(size_t)c * lanes] = y[c];
    out[(size_t)A.n_ch * lanes] = g;
}

// ---- carry: one thread per (symbol, chain), serial over the tiles ------------------------------------------------------------
// grid.y = chain (n_ch = the MACD signal line).  The loop-carried work is one fma per tile; the loads of B_k are issued
// LR_CB tiles ahead.  Results go to a second array (`carry`): the signal line's thread re-derives the fast / slow states
// it needs from the same B_k values the chain threads read.
constexpr int LR_CB = 16;
__global__ void __launch_bounds__(64) lr_carry_kernel(const __grid_constant__ LongArgs A) {
    const size_t lanes = (size_t)A.n_blocks * SYM;
    const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int c = blockIdx.y;
    if (s >= lanes) return;
    const size_t stride = (size_t)(A.n_ch + 1) * lanes;
    if (c < A.n_ch) {
        const int seed_tile = (A.p[c] - 1) / A.L;
        const double Ac = A.A[c];
        const double *in = A.agg + (size_t)c * lanes + s;
        double *out = A.carry + (size_t)c * lanes + s;
        double y = 0.0;
        for (int tb = 0; tb < A.n_tiles; tb += LR_CB) {
            double bk[LR_CB];
#pragma unroll
            for (int i = 0; i < LR_CB; ++i) bk[i] = (tb + i < A.n_tiles) ? __ldcg(in + (size_t)(tb + i) * stride) : 0.0;
#pragma unroll
            for (int i = 0; i < LR_CB; ++i) {
                const int tt = tb + i;
                if (tt >= A.n_tiles) break;
                if (tt < seed_tile) y = 0.0;
                else if (tt == seed_tile) y = bk[i];                         // the tile that holds the seed bar starts from the seed
                else y = fma(Ac, y, bk[i]);
                out[(size_t)tt * stride] = y;
            }
        }
        return;
    }
    if (!A.macd) return;
    // the signal line: it needs the fast / slow states at the START of each tile.  With f_j = f_loc_j + af^(j+1) f0 (and the
    // same for s), dif_j = dif_loc_j + af^(j+1) f0 - as^(j+1) s0, and the signal's end state is linear in its inputs:
    // g_end = Ag g0 + g_loc_end + Cf f0 - Cs s0, Cf = alpha_g * sum_j (1 - alpha_g)^(L-1-j) af^(j+1)
    const double *inf_ = A.agg + s, *ins = A.agg + lanes + s, *ing = A.agg + (size_t)A.n_ch * lanes + s;
    double *out = A.carry + (size_t)A.n_ch * lanes + s;
    double f = 0.0, sl = 0.0, g = 0.0;
    for (int tb = 0; tb < A.n_tiles; tb += LR_CB) {
        double bf[LR_CB], bs[LR_CB], bg[LR_CB];
#pragma unroll
        for (int i = 0; i < LR_CB; ++i) {
            const bool use = tb + i < A.n_tiles;
            bf[i] = use ? __ldcg(inf_ + (size_t)(tb + i) * stride) : 0.0;
            bs[i] = use ? __ldcg(ins + (size_t)(tb + i) * stride) : 0.0;
            bg[i] = use ? __ldcg(ing + (size_t)(tb + i) * stride) : 0.0;
        }
#pragma unroll
        for (int i = 0; i < LR_CB; ++i) {
            const int tt = tb + i;
            if (tt >= A.n_tiles) break;
            if (tt == 0) { g = bg[i]; f = bf[i]; sl = bs[i]; }               // (MACD periods fit tile 0: its end states are absolute)
            else {
                g = fma(A.A_g, g, bg[i]) + (A.Cf * f - A.Cs * sl);
                f = fma(A.A[0], f, bf[i]);
                sl = fma(A.A[1], sl, bs[i]);
            }
            out[(size_t)tt * stride] = g;
        }
    }
}

// ---- final: every output of one tile from the carried start state, in the reference's operation order ---------------------------
template <bool MACD>
__global__ void __launch_bounds__(128) lr_final_kernel(const __grid_constant__ LongArgs A) {
    const int lane = threadIdx.x & 31;
    const long long unit = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (unit >= (long long)A.n_tiles * A.n_blocks) return;
    const int tt = (int)(unit / A.n_blocks), b = (int)(unit % A.n_blocks);
    const int t0 = tt * A.L, t1 = min(t0 + A.L, A.n_bars);
    const size_t base = ((size_t)b * A.bars_padded + t0) * SYM + lane;
    const double *x = A.x + base;
    const size_t lanes = (size_t)A.n_blocks * SYM;
    const double *prev = A.carry + (size_t)(tt > 0 ? tt - 1 : 0) * (A.n_ch + 1) * lanes + b * SYM + lane;
    double y[LR_MAX_CH];
    int from[LR_MAX_CH];                   // first bar of the tile at which chain c runs its recurrence; its first value is at from - 1
#pragma unroll
    for (int c = 0; c < LR_MAX_CH; ++c) {
        y[c] = 0.0;
        from[c] = t0;
        if (c < A.n_ch) {
            const int ts = A.p[c] - 1;
            if (ts >= t1) from[c] = 0x7fffffff;                           // all null in this tile
            else if (ts >= t0) { from[c] = ts + 1; y[c] = A.seed[(size_t)c * lanes + b * SYM + lane]; }
            else y[c] = prev[(size_t)c * lanes];
        }
    }
    MacdHead head;
    double g = 0.0;
    if (MACD) { if (tt == 0) head.init(); else g = prev[(size_t)A.n_ch * lanes]; }
    const double nn = qnan();
    for (int tb = t0; tb < t1; tb += LR_BATCH) {
        double xv[LR_BATCH];
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) xv[i] = (tb + i < t1) ? ld_stream(x + (size_t)(tb - t0 + i) * SYM) : 0.0;
#pragma unroll
        for (int i = 0; i < LR_BATCH; ++i) {
            const int t = tb + i;
            if (t >= t1) break;
            const size_t o = base + (size_t)(t - t0) * SYM;
#pragma unroll
            for (int c = 0; c < LR_MAX_CH; ++c) {
                if (c >= A.n_ch) continue;
                if (t >= from[c]) y[c] = fma(A.alpha[c], xv[i] - y[c], y[c]);          // overlap.rs:698
                if (A.chain_out[c]) stg(A.chain_out[c] + o, (t >= from[c] - 1) ? y[c] : nn);
            }
            if (MACD) {
                double dif, sig;
                bool okd = true, okg = true;
                if (tt == 0) head.step(A, xv[i], t, dif, sig, okd, okg);
                else {
                    dif = y[0] - y[1];                                   // momentum.rs:264
                    g = fma(A.alpha_g, dif - g, g);
                    sig = g;
                }
                stg(A.macd_out[0] + o, okd ? dif : nn);
                stg(A.macd_out[1] + o, okg ? sig : nn);
                stg(A.macd_out[2] + o, (okd && okg) ? dif - sig : nn);   // :275
            }
        }
    }
}

}  // namespace pqb
