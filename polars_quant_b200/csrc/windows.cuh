// windows.cuh -- the rolling max / min suite over MANY windows in one launch (BASELINE config 5: KDJ(k) for k in
// 5 / 9 / 14 / 60 / 250, WILLR / MIDPRICE / Donchian(p) for p in 5 / 20 / 55 / 250, ATR(14) on 10,000 x 5,040).
//
// The fused suite kernel carries ONE period per indicator, so this set used to cost nine launches, each re-reading high /
// low / close and each latency-bound (two or three role warps per CTA).  Here every (indicator, window) pair is a UNIT;
// the host deals the units to G groups, CTA (b, g) runs group g's units (one warp each, lane = symbol, serial walk in the
// reference's operation order: every output bit-identical to the oracle) for symbol block b, fed by its own TMA producer
// warp over the same staged high / low / close bars.  More, smaller CTAs than one per symbol block: the grid (n_blocks x
// G) spreads evenly over the 148 SMs and an SM holds several CTAs, so the serial chains of many windows overlap.
//   KDJ(k, sk, sd)   momentum.py:178-186 + SURVEY D3: polars rolling max / min (full window), fastk, two calc_sma passes
//   WMD(p)           willr momentum.rs:630-662, midprice overlap.rs:281-404, Donchian upper / lower (SURVEY D3): one van
//                    Herk / Gil-Werman pair of arrays serves all four lines
//   ATR(p)           atr volatility.rs:18-31: calc_trange + calc_ema(trange, 2p - 1)
// van Herk arrays (p + 1 slots of 32 lanes per array) live in shared memory up to W_SMEM_MAX bars; longer windows use the
// two-level form (Ext2 below: 2 sqrt(p)-sized arrays in shared memory, raw rows re-read from the input planes by TMA).
// No producer warp: the unit warp that is LAST to leave a stage refills it (one shared-memory counter per stage), so every
// warp of the CTA computes and a CTA of U units costs U warps of registers.
// Null-aware variant (window_suite_kernel<..., true>, for the symbol blocks of a panel with halts, delistings or fields listed
// on different rows): each stage also carries the stage's input validity words, every unit walks the step_nulls() body of the
// suite role it mirrors (Role3 / Role5 / Role6 in suite_kernel.cuh) and every output line leaves one ballot word per bar.
#pragma once
#include "suite_kernel.cuh"

namespace pqb {

constexpr int W_MAX_UNITS = 6;        // unit warps per CTA
constexpr int W_MAX_TOTAL = 12;       // units per launch (6 KDJ windows + 5 WILLR / MIDPRICE / Donchian windows + ATR)
constexpr int W_MAX_GROUPS = W_MAX_TOTAL;
constexpr int W_SMEM_MAX = 32;        // windows up to this many bars keep one-level van Herk arrays (PQB_WIN_SMEM_MAX)
constexpr int W_FIELDS = 3;           // close, high, low
constexpr int W_STAGE_BYTES = W_FIELDS * SB * SYM * 8;      // 6 KB
constexpr int W_CTRL_BYTES = 128;     // NS full barriers, W_MAX_UNITS unit barriers (Ext2), NS stage counters
static_assert(NS * 8 + W_MAX_UNITS * 8 + NS * 4 <= W_CTRL_BYTES, "control area");

enum WinKind { WK_NONE = 0, WK_KDJ = 1, WK_WMD = 2, WK_ATR = 3 };

struct WinUnit {
    int kind, w;                       // window (KDJ fastk_period / WMD timeperiod / ATR timeperiod)
    int sk, sd;                        // KDJ smoothings (calc_sma periods)
    double inv_sk, inv_sd;             // 1.0 / p (overlap.rs:880)
    int ep;                            // ATR: 2p - 1 (volatility.rs:30)
    double alpha;                      // ATR: 2 / (ep + 1)
    int off_h, off_l;                  // one-level van Herk arrays (doubles from the ring area); two-level: off_h = its area, off_l = -1
    int seg;                           // two-level: segment length b (8 or 16)
    int piped;                         // software-pipelined steady path
    int off_fk, off_sk;                // KDJ: the two SMA windows
    double *out[4];                    // KDJ: K, D, J | WMD: willr, midprice, donchian_upper, donchian_lower | ATR: atr
};

struct WinArgs {
    const double *in[W_FIELDS];        // close, high, low (tiled planes)
    const int *start;                  // per-symbol first valid bar
    WinUnit u[W_MAX_TOTAL];            // group g's units are u[first[g] .. first[g] + n_units[g])
    int first[W_MAX_GROUPS];
    int n_units[W_MAX_GROUPS];
    int smem_bytes[W_MAX_GROUPS];
    int n_groups;
    int ns;                            // stages of the input ring (2 .. NS)
    int relaxed_wait;                  // sleep between failed tries of the stage wait
    int block_major;                   // CTA order: the groups of one symbol block next to each other (they share its input rows in L2)
    int steady_lead;                   // a lane is past every warm-up once t - start >= steady_lead
    int n_symbols, n_bars, n_blocks, bars_padded;   // (n_blocks: the blocks of this launch)
    const int *blist;                  // block i of the launch is blist[i] (nullptr: block i)
    // null-aware variant only
    const uint32_t *vmask;             // input validity words [block][bar][4] (pack_mask_kernel)
    const uint8_t *symflags;           // per symbol: bit f = field f has a null after its first valid bar
    uint32_t *ovm[W_MAX_TOTAL][4];     // unit i, line q: ballot words [block][bar]
    int mask_off;                      // shared-memory byte offset of the stage ring's validity words
};
constexpr int W_STAGE_MASK_BYTES = SB * N_IN * 4;    // one 32-lane word per bar and field

// Two-level van Herk / Gil-Werman for LONG windows (p > W_SMEM_MAX), entirely in shared memory.
// The one-level form (Ext) keeps p + 1 slots per array: the raw values of the current block of p bars, turned in place into
// the suffix extremes the NEXT block reads.  Here the block is cut into m segments of b bars and only three short arrays
// exist (2 b + m + 3 slots instead of p + 1: 50 instead of 251 for p = 250, b = 16):
//   A[0..m]   extremes of the current block's finished segments; at the block end a reverse scan turns them into
//             CHECKPOINTS: A[s] = extreme of segments s.. of that block (A[m] = sentinel).  In place: during block k, slot s
//             is rewritten at the end of segment s, after the checkpoint of the previous block in it was last needed;
//   buf[1..len] suffix extremes of ONE segment of the previous block, i.e. exactly the values Ext would read while the
//             current block walks through the same segment: buf[j] = max(raw[j..len-1], checkpoint of the next segment);
//   raw[0..b) the raw rows of the segment after that one, RE-READ from the panel's own tiled input plane (32 symbols x 8
//             bytes per bar, contiguous) by one TMA bulk copy per field, issued one segment (b bars) before they are needed.
// Nothing is written to global memory and nothing lives in L2: the first version kept p + 1-slot arrays in a global scratch
// (100 MB for config 5), which the 28 output streams evicted from L2 -- 21.5 GB of DRAM traffic for 12.5 GB of algorithmic
// bytes and an L2 / DRAM round trip on every bar's critical path (profiles/r02k_launch_summary.txt).
// max / min are exact, so the association (segments, checkpoints) does not change a bit of the result.
// LIVE (window_live_kernel): a walk may stop at any bar and a later launch resume from the saved object.  Such a walk
// issues no copy at init -- the rows of segment 0 may not exist yet -- and fetches them on entering block 0's last
// segment, when all of them have been walked; resume() re-issues the copy a saved walk had in flight.
template <bool LIVE = false>
struct Ext2T {
    uint32_t bh, bl, rh, rl, ah, al;   // byte offsets in shared memory (this lane's column; raw: the source lane's)
    uint32_t rdst, bar, phase;         // TMA destination (row 0 of raw high; raw low follows b rows later), this unit's mbarrier
    uint32_t roff, endoff;             // byte offset of slot r + 1 of buf; (len + 1) * 256
    const double *gh, *gl;             // this symbol block's high / low planes, bar 0
    int p, b, m, s, k, a, lane;        // window, segment length, segments per block; current segment, block index; first valid bar
    bool pending;                      // a bulk copy is in flight
    double ph, pl, sh, sl;             // prefix extremes of the current block / of its current segment
    __device__ __forceinline__ int seg_len(int seg) const { return (seg == m - 1) ? p - (m - 1) * b : b; }
    __device__ __forceinline__ void fetch(int t0, int len) {
        if (lane == 0) {
            const uint32_t bytes = (uint32_t)len * (SYM * 8);
            mbar_expect_tx(bar, 2 * bytes);
            tma_load_1d(rdst, gh + (size_t)t0 * SYM, bytes, bar);
            tma_load_1d(rdst + (uint32_t)b * (SYM * 8), gl + (size_t)t0 * SYM, bytes, bar);
        }
        pending = true;
    }
    // `area`: 2 (b + 1) + 2 b + 2 (m + 1) slots of 32 doubles; `mb`: this unit's mbarrier (initialised here)
    __device__ __forceinline__ void init(double *area, uint64_t *mb, const double *high, const double *low, int p_, int b_, int a_,
                                         int lane_, int src_lane, int bars_padded) {
        p = p_; b = b_; m = (p + b - 1) / b; a = a_; lane = lane_;
        double *q = area;
        bh = smem_off(q + lane); q += (b + 1) * SYM;
        bl = smem_off(q + lane); q += (b + 1) * SYM;
        rdst = smem_u32(q);
        rh = smem_off(q + src_lane); q += b * SYM;
        rl = smem_off(q + src_lane); q += b * SYM;
        ah = smem_off(q + lane); q += (m + 1) * SYM;
        al = smem_off(q + lane);
        gh = high; gl = low;
        for (int i = 0; i <= b; ++i) { sts(bh + i * (SYM * 8), vmin()); sts(bl + i * (SYM * 8), vmax()); }
        for (int i = 0; i <= m; ++i) { sts(ah + i * (SYM * 8), vmin()); sts(al + i * (SYM * 8), vmax()); }
        ph = sh = vmin();
        pl = sl = vmax();
        s = 0; k = 0; roff = SYM * 8; endoff = (uint32_t)(seg_len(0) + 1) * (SYM * 8);
        bar = smem_u32(mb); phase = 0; pending = false;
        if (lane == 0) { mbar_init(mb, 1); fence_mbar_init(); }
        __syncwarp();
        if (bars_padded >= p) fetch(0, seg_len(0));          // segment 0 of block 0: first needed when block 1 begins
    }
    __device__ __forceinline__ void finish() { if (pending) { mbar_wait(bar, phase); pending = false; } }   // never exit under a copy
    // Null-aware variant: `a` starts past every bar and becomes the first bar walked with high AND low valid (the validity
    // words fold explicit starts in).  A re-read raw row holds the intake's benign 1.0 under a null, not the -inf / +inf the
    // walked bar got.  No such row reaches a valid output:
    //  - rows before `a` are masked below, as in the plain kernel.  Every row segment_end() re-reads is older than the bar
    //    being walked, so `a` is final for it;
    //  - WILLR / MIDPRICE / Donchian: a symbol flagged in high or low has all-null lines, and an unflagged one has leading
    //    nulls only, so every row from `a` on is valid in both fields;
    //  - KDJ: a re-read row enters only the suffixes of bars whose window holds it, and fastk is null on every bar whose last
    //    k rows hold a null high or low (UnitKdj::step_nulls).
    // The checkpoints and the prefix extremes come from the walked bars, never from re-read rows.
    __device__ __forceinline__ void seen(int t, bool hl) { if (hl && t < a) a = t; }
    __device__ __forceinline__ void step(double h, double l, double &hn, double &ln) {
        ph = dmax(ph, h);
        pl = dmin(pl, l);
        sh = dmax(sh, h);
        sl = dmin(sl, l);
        hn = dmax(ph, lds(bh + roff));
        ln = dmin(pl, lds(bl + roff));
        roff += SYM * 8;
        if (roff == endoff) segment_end();
    }
    __device__ __forceinline__ void segment_end() {
        sts(ah + s * (SYM * 8), sh);
        sts(al + s * (SYM * 8), sl);
        sh = vmin();
        sl = vmax();
        if (++s == m) {                                    // block end: segment extremes -> checkpoints, newest to oldest
            double ch = vmin(), cl = vmax();
            for (int i = m - 1; i >= 0; --i) {
                ch = dmax(ch, lds(ah + i * (SYM * 8)));
                cl = dmin(cl, lds(al + i * (SYM * 8)));
                sts(ah + i * (SYM * 8), ch);
                sts(al + i * (SYM * 8), cl);
            }
            ph = vmin();
            pl = vmax();
            s = 0;
            ++k;
        }
        const int len = seg_len(s);
        roff = SYM * 8;
        endoff = (uint32_t)(len + 1) * (SYM * 8);
        if (k == 0) {                                      // no previous block yet: buf keeps its sentinels
            if constexpr (LIVE) { if (s == m - 1) fetch(0, seg_len(0)); }
            return;
        }
        // suffix extremes of segment s of block k - 1 from its raw rows, on top of the checkpoint of the segments after it
        mbar_wait(bar, phase);
        phase ^= 1;
        pending = false;
        const int t0 = (k - 1) * p + s * b;
        double ch = lds(ah + (s + 1) * (SYM * 8)), cl = lds(al + (s + 1) * (SYM * 8));
        sts(bh + len * (SYM * 8), ch);
        sts(bl + len * (SYM * 8), cl);
#pragma unroll 4
        for (int j = len - 1; j >= 1; --j) {
            const double xh = lds(rh + j * (SYM * 8)), xl = lds(rl + j * (SYM * 8));
            const bool in = t0 + j >= a;                   // bars before the symbol's first valid bar count as -inf / +inf
            ch = dmax(ch, in ? xh : ninf());
            cl = dmin(cl, in ? xl : pinf());
            sts(bh + j * (SYM * 8), ch);
            sts(bl + j * (SYM * 8), cl);
        }
        __syncwarp();                                      // every lane has read the raw rows: the next copy may overwrite them
        const int s2 = (s + 1 == m) ? 0 : s + 1;
        fetch(t0 + len, seg_len(s2));                      // segments are contiguous in time
    }
    // LIVE: continue a saved walk.  mbarrier phases and bulk copies end with their launch, so the unit's barrier starts
    // afresh (phase 0) and the copy the saved walk had in flight -- the rows the next segment_end() reads: segment s + 1 of
    // block k - 1, or segment 0 of block k from block k's last segment on -- is issued again.  A live walk has such a copy
    // in flight exactly when k >= 1 or s == m - 1 (the saved `pending` says nothing: finish() cleared it before the save).
    // Those rows lie 1 .. p - 1 bars before the walk's first bar (the host keeps at least p of them in front of the pushed
    // rows).  `high` / `low`: the planes' addresses of absolute bar 0.  The caller has put the raw rows' shared memory in
    // place (generic proxy).
    __device__ __forceinline__ void resume(uint64_t *mb, const double *high, const double *low) {
        gh = high; gl = low;
        bar = smem_u32(mb); phase = 0;
        if (lane == 0) {
            mbar_init(mb, 1);
            fence_mbar_init();
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        }
        __syncwarp();
        pending = false;
        if (k >= 1 || s == m - 1) {
            const int s2 = (s + 1 == m) ? 0 : s + 1;
            fetch((s + 1 == m) ? k * p : (k - 1) * p + s2 * b, seg_len(s2));
        }
    }
};
using Ext2 = Ext2T<false>;

__device__ __forceinline__ void seen(Ext &, int, bool) {}                   // (the one-level arrays hold walked bars only)
template <bool L>
__device__ __forceinline__ void seen(Ext2T<L> &e, int t, bool hl) { e.seen(t, hl); }

struct WCtx {
    size_t pos;        // element offset of (this lane, current bar)
    int a, n_bars;     // this lane's first valid bar; bars of the panel
    size_t mpos;       // null-aware variant: block * bars_padded + bar (ballot words)
    unsigned flags;    // null-aware variant: this lane's symbol flags
};

// null-aware variant: value (NaN when null) + the warp's validity word of this bar; called by all 32 lanes together
__device__ __forceinline__ void emitw(const WCtx &X, double *out, uint32_t *ovm, double v, bool ok) {
    const unsigned m = __ballot_sync(FULL, ok);
    stg(out + X.pos, ok ? v : qnan());
    if ((threadIdx.x & 31) == 0) ovm[X.mpos] = m;
}
// live walks: the prime walk over a history stores nothing (store = 0)
struct WCtxLive : WCtx {
    bool store;
};
__device__ __forceinline__ void emitw(const WCtxLive &X, double *out, uint32_t *ovm, double v, bool ok) {
    if (X.store) emitw(static_cast<const WCtx &>(X), out, ovm, v, ok);
}

// ---- KDJ(k, sk, sd) ---------------------------------------------------------------------------------------------------------
template <class EXT, bool PIPED>
struct UnitKdj {
    EXT ek;
    Ring fr, sr;
    double s_k, s_d;
    struct { int w, sk, sd; double inv_sk, inv_sd; double *out[3]; } U;      // this unit's parameters, in registers
    __device__ __forceinline__ void take(const WinUnit &u) {
        U.w = u.w; U.sk = u.sk; U.sd = u.sd; U.inv_sk = u.inv_sk; U.inv_sd = u.inv_sd;
        U.out[0] = u.out[0]; U.out[1] = u.out[1]; U.out[2] = u.out[2];
    }
    template <bool STEADY>
    __device__ __forceinline__ void step(const WCtx &X, int t, double c, double h, double l) {
        const int j = t - X.a;
        const bool live = STEADY || t < X.n_bars;
        const bool in = STEADY || (j >= 0 && live);
        const double nn = qnan();
        double hn, ln;
        ek.step(in ? h : ninf(), in ? l : pinf(), hn, ln);
        double ok_ = nn, od = nn, oj = nn;
        const int j1 = j - (U.w - 1);                     // index in the fastk series (polars rolling: k-1 nulls)
        const bool v1 = STEADY || (j1 >= 0 && live);
        // momentum.py:183 -- IEEE x / 0 (= x * inf: +-inf, or NaN for 0 / 0) without the slow path
        const double num = (c - ln) * 100.0, den = hn - ln;
        const double fk = (den == 0.0) ? num * copysign(pinf(), den) : num / den;
        const double oldf = fr.swap(fk);
        double sk = 0.0;
        const int j2 = j1 - (U.sk - 1);
        if (v1) {
            s_k += fk;                                    // slowk = calc_sma(fastk, sk) overlap.rs:871
            if (STEADY || j1 >= U.sk) s_k -= oldf;
            sk = s_k * U.inv_sk;
        }
        const double olds = sr.swap(sk);
        if (v1 && (STEADY || j2 >= 0)) {
            ok_ = sk;
            s_d += sk;                                    // slowd = calc_sma(slowk, sd)
            if (STEADY || j2 >= U.sd) s_d -= olds;
            if (STEADY || j2 >= U.sd - 1) {
                const double sd = s_d * U.inv_sd;
                od = sd;
                oj = 3.0 * sk - 2.0 * sd;                 // J = 3K - 2D (D3)
            }
        }
        stg(U.out[0] + X.pos, ok_);
        stg(U.out[1] + X.pos, od);
        stg(U.out[2] + X.pos, oj);
    }
    // ---- null-aware bar: Role5::step_nulls.  vb bit f = field f of this lane is valid at bar t.  polars' rolling max / min
    // are positional with a full window (fastk null unless close is valid and the last k rows are valid in high and in low);
    // the two calc_sma passes skip null inputs.  Flags do not kill KDJ.
    int run_h, run_l, nfk, nsk;
    uint32_t *ovm[3];
    template <class CX>
    __device__ __forceinline__ void step_nulls(const CX &X, int t, double c, double h, double l, unsigned vb) {
        const bool vc = vb & F_C, vh = vb & F_H, vl = vb & F_L;
        seen(ek, t, vh && vl);
        double hn, ln;
        ek.step(vh ? h : ninf(), vl ? l : pinf(), hn, ln);
        run_h = vh ? min(run_h + 1, 1 << 30) : 0;        // rows since the last null, separately for high and low
        run_l = vl ? min(run_l + 1, 1 << 30) : 0;
        const bool vfk = vc && run_h >= U.w && run_l >= U.w;
        bool okk = false, okd = false;
        double sk = 0.0, sd = 0.0;
        if (vfk) {
            const double num = (c - ln) * 100.0, den = hn - ln;
            const double fk = (den == 0.0) ? num * copysign(pinf(), den) : num / den;
            const int j1 = nfk++;
            const double oldf = fr.swap(fk);
            s_k += fk;
            if (j1 >= U.sk) s_k -= oldf;
            if (j1 >= U.sk - 1) {
                sk = s_k * U.inv_sk;
                okk = true;
                const int j2 = nsk++;
                const double olds = sr.swap(sk);
                s_d += sk;
                if (j2 >= U.sd) s_d -= olds;
                if (j2 >= U.sd - 1) {
                    sd = s_d * U.inv_sd;
                    okd = true;
                }
            }
        }
        emitw(X, U.out[0], ovm[0], sk, okk);
        emitw(X, U.out[1], ovm[1], sd, okd);
        emitw(X, U.out[2], ovm[2], 3.0 * sk - 2.0 * sd, okd);
    }
    __device__ __forceinline__ void finish() { ek.finish(); }
    // ---- software-pipelined steady bar (Role5::pipe of the suite kernel): A = window extremes of bar t, B = fastk's division
    // of bar t-1, C = the two running means and J of bar t-2.  The stages touch disjoint state, so the compiler overlaps the
    // three dependent chains of one loop iteration; each stage still sees every bar once, in order: same bits as step().
    static constexpr int DEPTH = PIPED ? 2 : 0;
    double pNum, pDen, pFk;
    template <int M>
    __device__ __forceinline__ void pipe(const WCtx &X, double c, double h, double l) {
        bool ok = true, z = false;
        double fk = 0.0, den = 1.0, num_n = 0.0, den_n = 0.0;
        if (M & 4) {
            const double oldf = fr.swap(pFk);
            s_k += pFk;                                   // slowk = calc_sma(fastk, sk) overlap.rs:871
            s_k -= oldf;
            const double sk = s_k * U.inv_sk;
            const double olds = sr.swap(sk);
            s_d += sk;                                    // slowd = calc_sma(slowk, sd)
            s_d -= olds;
            const double sd = s_d * U.inv_sd;
            const size_t q = X.pos - 2 * SYM;
            stg(U.out[0] + q, sk);
            stg(U.out[1] + q, sd);
            stg(U.out[2] + q, 3.0 * sk - 2.0 * sd);       // J = 3K - 2D (D3)
        }
        if (M & 2) {
            z = pDen == 0.0;
            den = z ? 1.0 : pDen;
            fk = div_fast(pNum, den, ok);
        }
        if (M & 1) {
            double hn, ln;
            ek.step(h, l, hn, ln);
            num_n = (c - ln) * 100.0;                     // momentum.py:183
            den_n = hn - ln;
        }
        if (M & 2) {
            if (!ok) fk = (pNum == 0.0) ? pNum * den : slow_div(pNum, den);
            pFk = z ? pNum * copysign(pinf(), pDen) : fk;
        }
        if (M & 1) {
            pNum = num_n;
            pDen = den_n;
        }
    }
};

// ---- WILLR / MIDPRICE / Donchian(p) -----------------------------------------------------------------------------------------
template <class EXT, bool PIPED>
struct UnitWmd {
    EXT ew;
    struct { int w; double *out[4]; } U;
    __device__ __forceinline__ void take(const WinUnit &u) {
        U.w = u.w;
        for (int q = 0; q < 4; ++q) U.out[q] = u.out[q];
    }
    template <bool STEADY>
    __device__ __forceinline__ void step(const WCtx &X, int t, double c, double h, double l) {
        const int j = t - X.a;
        const bool live = STEADY || t < X.n_bars;
        const bool in = STEADY || (j >= 0 && live);
        const double nn = qnan();
        double hn, ln;
        ew.step(in ? h : ninf(), in ? l : pinf(), hn, ln);
        if (U.out[0]) {                                   // willr momentum.rs:630-662
            double o = nn;
            if ((STEADY || j >= U.w - 1) && live) {
                const double diff = hn - ln;
                const bool z = diff == 0.0;
                const double q = -100.0 * (hn - c) / (z ? 1.0 : diff);                    // :653-657
                o = z ? 0.0 : q;
            }
            stg(U.out[0] + X.pos, o);
        }
        if (U.out[1]) stg(U.out[1] + X.pos, in ? (hn + ln) / 2.0 : nn);                   // midprice overlap.rs:401
        if (U.out[2]) stg(U.out[2] + X.pos, in ? hn : nn);                                // Donchian upper / lower (D3)
        if (U.out[3]) stg(U.out[3] + X.pos, in ? ln : nn);
    }
    // ---- null-aware bar: Role6::step_nulls.  The window advances on every bar; a bar without both high and low enters it as
    // -inf / +inf.  willr is all-null for a symbol flagged in close, high or low, and otherwise valid where close, high and
    // low are, after p - 1 earlier bars with high and low valid; midprice and the Donchian lines are all-null for a symbol
    // flagged in high or low, and otherwise valid where high and low are.
    int n_valid;
    uint32_t *ovm[4];
    template <class CX>
    __device__ __forceinline__ void step_nulls(const CX &X, int t, double c, double h, double l, unsigned vb) {
        const bool in = (vb & F_H) && (vb & F_L);
        seen(ew, t, in);
        double hn, ln;
        ew.step(in ? h : ninf(), in ? l : pinf(), hn, ln);
        if (U.out[0]) {                                   // willr momentum.rs:630-662
            const bool ok = !(X.flags & (F_C | F_H | F_L)) && in && (vb & F_C) && n_valid >= U.w - 1;
            const double diff = hn - ln;
            const bool z = diff == 0.0;
            const double q = -100.0 * (hn - c) / (z ? 1.0 : diff);
            emitw(X, U.out[0], ovm[0], z ? 0.0 : q, ok);
        }
        const bool v = in && !(X.flags & (F_H | F_L));
        if (U.out[1]) emitw(X, U.out[1], ovm[1], (hn + ln) / 2.0, v);                   // midprice overlap.rs:401
        if (U.out[2]) emitw(X, U.out[2], ovm[2], hn, v);                                // Donchian upper / lower (D3)
        if (U.out[3]) emitw(X, U.out[3], ovm[3], ln, v);
        n_valid += in ? 1 : 0;
    }
    __device__ __forceinline__ void finish() { ew.finish(); }
    // ---- software-pipelined steady bar (Role6::pipe): A = window extremes, midprice and the Donchian lines of bar t,
    // B = willr's division of bar t-1
    static constexpr int DEPTH = PIPED ? 1 : 0;
    double pH, pL, pC;
    template <int M>
    __device__ __forceinline__ void pipe(const WCtx &X, double c, double h, double l) {
        bool ok = true, z = false;
        double q = 0.0, den = 1.0, num = 0.0, wh = 0.0, wl = 0.0;
        if (M & 2) {
            const double diff = pH - pL;
            z = diff == 0.0;
            den = z ? 1.0 : diff;
            num = -100.0 * (pH - pC);                                                     // momentum.rs:653-657
            q = div_fast(num, den, ok);
        }
        if (M & 1) {
            ew.step(h, l, wh, wl);
            stg(U.out[1] + X.pos, (wh + wl) / 2.0);                                       // midprice overlap.rs:401
            stg(U.out[2] + X.pos, wh);                                                    // Donchian upper / lower (D3)
            stg(U.out[3] + X.pos, wl);
        }
        if (M & 2) {
            if (!ok) q = (num == 0.0) ? num * den : slow_div(num, den);
            stg(U.out[0] + X.pos - SYM, z ? 0.0 : q);
        }
        if (M & 1) {
            pH = wh;
            pL = wl;
            pC = c;
        }
    }
};

// ---- ATR(p) -------------------------------------------------------------------------------------------------------------------
struct UnitAtr {
    Ema atr;
    double pc;
    struct { int ep; double alpha; double *out[1]; } U;
    __device__ __forceinline__ void take(const WinUnit &u) { U.ep = u.ep; U.alpha = u.alpha; U.out[0] = u.out[0]; }
    template <bool STEADY>
    __device__ __forceinline__ void step(const WCtx &X, int t, double c, double h, double l) {
        const int j = t - X.a;
        const bool live = STEADY || t < X.n_bars;
        const double tr = rs_max(rs_max(h - l, fabs(h - pc)), fabs(l - pc));             // volatility.rs:77
        const bool ok = atr.step<STEADY>(tr, j - 1, U.ep, U.alpha);                      // :30 calc_ema(trange, 2p-1)
        stg(U.out[0] + X.pos, (ok && live) ? atr.y : qnan());
        pc = c;
    }
    // ---- null-aware bar: Role3::step_nulls.  calc_trange's close.shift(1) is positional: the true range is valid where high
    // and low are valid and the previous ROW's close is; calc_ema counts valid true ranges only.  Flags do not kill ATR.
    int n_tr;
    bool pcv;
    uint32_t *ovm[1];
    template <class CX>
    __device__ __forceinline__ void step_nulls(const CX &X, int t, double c, double h, double l, unsigned vb) {
        const bool vtr = t >= 1 && (vb & F_H) && (vb & F_L) && pcv;
        const double tr = rs_max(rs_max(h - l, fabs(h - pc)), fabs(l - pc));             // volatility.rs:77
        const bool ok = atr.step<false>(tr, vtr ? n_tr : -1, U.ep, U.alpha);
        emitw(X, U.out[0], ovm[0], atr.y, ok);
        n_tr += vtr ? 1 : 0;
        pc = c;
        pcv = vb & F_C;
    }
    __device__ __forceinline__ void finish() {}
    static constexpr int DEPTH = 0;
    template <int M>
    __device__ __forceinline__ void pipe(const WCtx &, double, double, double) {}
};

// Live window panels (windows_live_host.inc): a walk covers the absolute bars [t_base, A.n_bars).  The input planes are
// [block][in_stride][32] with the walk's first bar at A.in[f] (row `tail` of each block: the high / low rows before it stay
// readable for Ext2's re-reads); outputs and validity words are [block][A.bars_padded] from the walk's first bar.  The
// state of CTA (block, group) is the unit objects (word i of unit warp u, lane l at (u * W_LIVE_UNIT_WORDS + i) * 32 + l)
// followed by the CTA's ring area.
struct WinLiveArgs {
    unsigned long long *state;         // [n_blocks][n_groups][group_words]
    long long group_words;             // W_MAX_UNITS * W_LIVE_UNIT_WORDS * 32 + ring_bytes / 8
    int ring_bytes;                    // the largest group's ring area (smem_bytes minus stages and control area)
    int t_base;                        // absolute index of the walk's first bar
    int in_stride;                     // rows per symbol block of the input planes
    int prime;                         // 1: the units start from init() and store nothing; 0: they resume from the state
    int commit;                        // 1: the walk's end state is written back
};

// (NULLS: stage st's validity words are at byte A.mask_off + st * W_STAGE_MASK_BYTES of the shared memory)
template <bool NULLS, class UNIT, bool LIVE = false>
__device__ __forceinline__ void run_unit(UNIT &R, const WinArgs &A, const WinUnit &U_, uint32_t stage, uint32_t full, int *cnt,
                                         int n_units, int block, int lane, int a, const WinLiveArgs *L = nullptr) {
    R.take(U_);
    const int sym = block * SYM + lane;
    const int src_lane = (sym < A.n_symbols) ? lane : 0;   // lanes past the last symbol follow lane 0 (no slow-path divisions)
    std::conditional_t<LIVE, WCtxLive, WCtx> X{WCtx{(size_t)block * A.bars_padded * SYM + lane, a, A.n_bars}};
    if constexpr (LIVE) X.store = !L->prime;
    if constexpr (NULLS) {
        X.mpos = (size_t)block * A.bars_padded;
        X.flags = A.symflags[(sym < A.n_symbols) ? sym : block * SYM];
    }
    int amax = a;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) amax = max(amax, __shfl_xor_sync(FULL, amax, d));
    const long long steady_from = (long long)amax + A.steady_lead;
    const int n_iter = A.bars_padded / SB;
    const size_t base = (size_t)block * A.bars_padded * SYM;
    const size_t ibase = LIVE ? (size_t)block * L->in_stride * SYM : base;   // (input planes)
    const int ns = A.ns;
    // software-pipelined steady path: `fill` = primed pipeline stages (warp-uniform); drained before any general bar
    constexpr int DEPTH = UNIT::DEPTH, PIPE_ALL = (1 << (DEPTH + 1)) - 1;
    int fill = 0;
    auto drain = [&]() {                                   // X.pos = the next unprocessed bar
        if constexpr (DEPTH == 2) {
            R.template pipe<6>(X, 0.0, 0.0, 0.0);
            X.pos += SYM;
            R.template pipe<4>(X, 0.0, 0.0, 0.0);
            X.pos -= SYM;
        } else if constexpr (DEPTH == 1) {
            R.template pipe<2>(X, 0.0, 0.0, 0.0);
        }
        fill = 0;
    };
    for (int it = 0; it < n_iter; ++it) {
        const int st = it % ns;
        if (A.relaxed_wait) mbar_wait_relaxed(full + st * 8, (it / ns) & 1);
        else mbar_wait(full + st * 8, (it / ns) & 1);
        const uint32_t sp = st * W_STAGE_BYTES + src_lane * 8;
        const int t0 = (LIVE ? L->t_base : 0) + it * SB;
        if constexpr (NULLS) {
            // (no software pipelining, no fast stages; bars past the panel's end leave the state as it is)
            const uint32_t mp = stage + (uint32_t)A.mask_off + st * W_STAGE_MASK_BYTES;
#pragma unroll 1
            for (int b = 0; b < SB; ++b) {
                if (t0 + b < A.n_bars) {
                    const uint32_t q = sp + b * (SYM * 8);
                    uint4 mw;
                    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(mw.x), "=r"(mw.y), "=r"(mw.z), "=r"(mw.w) : "r"(mp + b * 16));
                    // (a ragged block's spare lanes follow lane 0's validity too)
                    const unsigned vb = ((mw.x >> src_lane) & 1u) | (((mw.y >> src_lane) & 1u) << 1) | (((mw.z >> src_lane) & 1u) << 2);
                    R.step_nulls(X, t0 + b, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8), vb);
                }
                X.pos += SYM;
                X.mpos += 1;
            }
        } else if (t0 >= steady_from && t0 + SB <= A.n_bars) {
            int b = 0;
            if constexpr (DEPTH > 0) {
                for (; fill < DEPTH; ++fill, ++b) {        // prime: stage A alone, then A + B
                    const uint32_t q = sp + b * (SYM * 8);
                    if (fill == 0) R.template pipe<1>(X, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8));
                    else R.template pipe<3>(X, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8));
                    X.pos += SYM;
                }
            }
#pragma unroll 1
            for (; b < SB; ++b) {
                const uint32_t q = sp + b * (SYM * 8);
                if constexpr (DEPTH > 0) R.template pipe<PIPE_ALL>(X, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8));
                else R.template step<true>(X, t0 + b, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8));
                X.pos += SYM;
            }
        } else {
            if constexpr (DEPTH > 0) { if (fill) drain(); }
#pragma unroll 1
            for (int b = 0; b < SB; ++b) {
                if (t0 + b < A.n_bars) {
                    const uint32_t q = sp + b * (SYM * 8);
                    R.template step<false>(X, t0 + b, lds(q), lds(q + 1 * SB * SYM * 8), lds(q + 2 * SB * SYM * 8));
                }
                X.pos += SYM;
            }
        }
        __syncwarp();
        // the last unit warp to leave the stage refills it with the bars of iteration it + NS
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(&cnt[st], 1) == n_units - 1) {
                atomicExch(&cnt[st], 0);
                const int nx = it + ns;
                if (nx < n_iter) {
                    mbar_expect_tx(full + st * 8, (uint32_t)W_STAGE_BYTES + (NULLS ? W_STAGE_MASK_BYTES : 0));
                    const size_t off = ibase + (size_t)nx * SB * SYM;
#pragma unroll
                    for (int f = 0; f < W_FIELDS; ++f)
                        tma_load_1d(stage + st * W_STAGE_BYTES + f * SB * SYM * 8, A.in[f] + off, (uint32_t)(SB * SYM * sizeof(double)),
                                    full + st * 8);
                    if constexpr (NULLS)
                        tma_load_1d(stage + (uint32_t)A.mask_off + st * W_STAGE_MASK_BYTES, A.vmask + (base / SYM + (size_t)nx * SB) * N_IN,
                                    W_STAGE_MASK_BYTES, full + st * 8);
                }
            }
        }
    }
    if constexpr (DEPTH > 0) { if (fill) drain(); }
    R.finish();
}

// ---- live walks: unit objects and the CTA's ring area <-> the state buffer ----------------------------------------------------
static_assert(std::is_trivially_copyable<UnitKdj<Ext, false>>::value && std::is_trivially_copyable<UnitKdj<Ext2T<true>, false>>::value &&
              std::is_trivially_copyable<UnitWmd<Ext, false>>::value && std::is_trivially_copyable<UnitWmd<Ext2T<true>, false>>::value &&
              std::is_trivially_copyable<UnitAtr>::value, "a unit object is saved and restored as raw bytes");
constexpr size_t w_max(size_t a, size_t b) { return a > b ? a : b; }
constexpr int W_LIVE_UNIT_WORDS = (int)(w_max(w_max(w_max(sizeof(UnitKdj<Ext, false>), sizeof(UnitKdj<Ext2T<true>, false>)),
                                                   w_max(sizeof(UnitWmd<Ext, false>), sizeof(UnitWmd<Ext2T<true>, false>))),
                                             sizeof(UnitAtr)) + 7) / 8;

// a unit object <-> its words (lane-interleaved: a warp moves 256 contiguous bytes per word)
template <bool LOAD, class UNIT>
__device__ __forceinline__ void win_live_unit(UNIT &R, unsigned long long *uw, int lane) {
    static_assert(sizeof(UNIT) % 8 == 0, "unit objects are saved in 8-byte words");
    constexpr int W = (int)(sizeof(UNIT) / 8);
    unsigned long long w[W];
    if (!LOAD) __builtin_memcpy(w, &R, sizeof(UNIT));
#pragma unroll
    for (int i = 0; i < W; ++i) {
        if (LOAD) w[i] = uw[(size_t)i * SYM + lane];
        else uw[(size_t)i * SYM + lane] = w[i];
    }
    if (LOAD) __builtin_memcpy(&R, w, sizeof(UNIT));
}

// the CTA's ring area <-> the state buffer: the unit warps' threads move 16-byte pieces
template <bool LOAD>
__device__ __forceinline__ void win_live_rings(double *rings, unsigned long long *grp, int ring_bytes, int n_threads) {
    uint4 *g = reinterpret_cast<uint4 *>(grp + (size_t)W_MAX_UNITS * W_LIVE_UNIT_WORDS * SYM);
    uint4 *s = reinterpret_cast<uint4 *>(rings);
    for (int u = threadIdx.x; u < ring_bytes / 16; u += n_threads) {
        if (LOAD) s[u] = g[u];
        else g[u] = s[u];
    }
}

// grid = n_blocks * n_groups, blockDim = 32 * (the largest group's units); CTA (b, g): warp i = unit i of group g.
// Two builds: <128, 4> for up to four units per CTA (118 registers, nothing spilled: at 96 the pipelined loops spill and
// the launch is slower, profiles/r02p_window_sweep.txt), <192, 2> for five or six.  NULLS: the null-aware variant (blocks
// with a flagged symbol; A.start unused, the validity words carry the starts).
template <int MAXT, int MINB, bool NULLS = false>
__global__ void __launch_bounds__(MAXT, MINB) window_suite_kernel(const __grid_constant__ WinArgs A) {
    uint64_t *full_p = reinterpret_cast<uint64_t *>(smem_dyn + A.ns * W_STAGE_BYTES);
    uint64_t *unit_p = full_p + NS;
    int *cnt = reinterpret_cast<int *>(unit_p + W_MAX_UNITS);
    double *rings = reinterpret_cast<double *>(smem_dyn + A.ns * W_STAGE_BYTES + W_CTRL_BYTES);
    const uint32_t stage = smem_u32(smem_dyn), full = smem_u32(full_p);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // group-major: the CTAs of the heaviest group (group 0) are scheduled first, the lighter groups fill in behind them
    const int g = A.block_major ? (int)(blockIdx.x % (unsigned)A.n_groups) : (int)(blockIdx.x / (unsigned)A.n_blocks);
    const int bi = A.block_major ? (int)(blockIdx.x / (unsigned)A.n_groups) : (int)(blockIdx.x % (unsigned)A.n_blocks);
    const int block = A.blist ? A.blist[bi] : bi;
    const int n_units = A.n_units[g];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full_p[s], 1);         // (NS slots exist in the control area whatever A.ns is)
            cnt[s] = 0;
        }
        fence_mbar_init();
        const int n_iter = A.bars_padded / SB;
        const size_t base = (size_t)block * A.bars_padded * SYM;
        for (int it = 0; it < A.ns && it < n_iter; ++it) {
            mbar_expect_tx(full + it * 8, (uint32_t)W_STAGE_BYTES + (NULLS ? W_STAGE_MASK_BYTES : 0));
#pragma unroll
            for (int f = 0; f < W_FIELDS; ++f)
                tma_load_1d(stage + it * W_STAGE_BYTES + f * SB * SYM * 8, A.in[f] + base + (size_t)it * SB * SYM,
                            (uint32_t)(SB * SYM * sizeof(double)), full + it * 8);
            if constexpr (NULLS)
                tma_load_1d(stage + (uint32_t)A.mask_off + it * W_STAGE_MASK_BYTES, A.vmask + ((size_t)block * A.bars_padded + (size_t)it * SB) * N_IN,
                            W_STAGE_MASK_BYTES, full + it * 8);
        }
    }
    __syncthreads();
    if (warp >= n_units) return;
    const WinUnit &U = A.u[A.first[g] + warp];
    uint32_t *const *ovm = A.ovm[A.first[g] + warp];
    const int sym = block * SYM + lane;
    const int a = (!NULLS && A.start) ? A.start[(sym < A.n_symbols) ? sym : block * SYM] : 0;
    const int src_lane = (sym < A.n_symbols) ? lane : 0;
    const size_t pbase = (size_t)block * A.bars_padded * SYM;
    auto kdj = [&](auto &R) {
        R.fr.init(rings + U.off_fk, U.sk, lane);
        R.sr.init(rings + U.off_sk, U.sd, lane);
        R.s_k = R.s_d = 0.0;
        R.pNum = R.pDen = R.pFk = 0.0;
        if constexpr (NULLS) {
            R.run_h = R.run_l = R.nfk = R.nsk = 0;
            for (int q = 0; q < 3; ++q) R.ovm[q] = ovm[q];
        }
        __syncwarp();
        run_unit<NULLS>(R, A, U, stage, full, cnt, n_units, block, lane, a);
    };
    auto wmd = [&](auto &R) {
        R.pH = R.pL = R.pC = 0.0;
        if constexpr (NULLS) {
            R.n_valid = 0;
            for (int q = 0; q < 4; ++q) R.ovm[q] = ovm[q];
        }
        __syncwarp();
        run_unit<NULLS>(R, A, U, stage, full, cnt, n_units, block, lane, a);
    };
    auto one = [&](auto &R) { R.init(rings + U.off_h, rings + U.off_l, U.w, lane); };
    // (NULLS: the first bar with high and low valid is found on the walk, Ext2::seen)
    auto two = [&](auto &R) { R.init(rings + U.off_h, unit_p + warp, A.in[1] + pbase, A.in[2] + pbase, U.w, U.seg, NULLS ? INT_MAX : a, lane, src_lane, A.bars_padded); };
    // (the null-aware variant has no software-pipelined path)
    if (U.kind == WK_KDJ) {
        if (U.off_l >= 0) {
            if (!NULLS && U.piped) { UnitKdj<Ext, true> R; one(R.ek); kdj(R); } else { UnitKdj<Ext, false> R; one(R.ek); kdj(R); }
        } else {
            if (!NULLS && U.piped) { UnitKdj<Ext2, true> R; two(R.ek); kdj(R); } else { UnitKdj<Ext2, false> R; two(R.ek); kdj(R); }
        }
    } else if (U.kind == WK_WMD) {
        if (U.off_l >= 0) {
            if (!NULLS && U.piped) { UnitWmd<Ext, true> R; one(R.ew); wmd(R); } else { UnitWmd<Ext, false> R; one(R.ew); wmd(R); }
        } else {
            if (!NULLS && U.piped) { UnitWmd<Ext2, true> R; two(R.ew); wmd(R); } else { UnitWmd<Ext2, false> R; two(R.ew); wmd(R); }
        }
    } else {
        UnitAtr R;
        R.atr.init();
        R.pc = 0.0;
        if constexpr (NULLS) {
            R.n_tr = 0;
            R.pcv = false;
            R.ovm[0] = ovm[0];
        }
        run_unit<NULLS>(R, A, U, stage, full, cnt, n_units, block, lane, a);
    }
}

// live window panels: the null-aware walk of every symbol block, resumable (WinLiveArgs).  The stage ring is the null-aware
// kernel's; the input planes are [block][L.in_stride][32].  (Its own kernel rather than a template flag of the one above:
// moving that kernel's body into a shared function changes the register assignment of the plain builds.)
template <int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) window_live_kernel(const __grid_constant__ WinArgs A, const __grid_constant__ WinLiveArgs Lv) {
    const WinLiveArgs *L = &Lv;
    uint64_t *full_p = reinterpret_cast<uint64_t *>(smem_dyn + A.ns * W_STAGE_BYTES);
    uint64_t *unit_p = full_p + NS;
    int *cnt = reinterpret_cast<int *>(unit_p + W_MAX_UNITS);
    double *rings = reinterpret_cast<double *>(smem_dyn + A.ns * W_STAGE_BYTES + W_CTRL_BYTES);
    const uint32_t stage = smem_u32(smem_dyn), full = smem_u32(full_p);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = A.block_major ? (int)(blockIdx.x % (unsigned)A.n_groups) : (int)(blockIdx.x / (unsigned)A.n_blocks);
    const int block = A.block_major ? (int)(blockIdx.x / (unsigned)A.n_groups) : (int)(blockIdx.x % (unsigned)A.n_blocks);
    const int n_units = A.n_units[g];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            mbar_init(&full_p[s], 1);
            cnt[s] = 0;
        }
        fence_mbar_init();
        const int n_iter = A.bars_padded / SB;
        const size_t ibase = (size_t)block * L->in_stride * SYM;
        for (int it = 0; it < A.ns && it < n_iter; ++it) {
            mbar_expect_tx(full + it * 8, (uint32_t)(W_STAGE_BYTES + W_STAGE_MASK_BYTES));
#pragma unroll
            for (int f = 0; f < W_FIELDS; ++f)
                tma_load_1d(stage + it * W_STAGE_BYTES + f * SB * SYM * 8, A.in[f] + ibase + (size_t)it * SB * SYM,
                            (uint32_t)(SB * SYM * sizeof(double)), full + it * 8);
            tma_load_1d(stage + (uint32_t)A.mask_off + it * W_STAGE_MASK_BYTES, A.vmask + ((size_t)block * A.bars_padded + (size_t)it * SB) * N_IN,
                        W_STAGE_MASK_BYTES, full + it * 8);
        }
    }
    __syncthreads();
    if (warp >= n_units) return;
    const WinUnit &U = A.u[A.first[g] + warp];
    uint32_t *const *ovm = A.ovm[A.first[g] + warp];
    const int sym = block * SYM + lane;
    const int src_lane = (sym < A.n_symbols) ? lane : 0;
    const int a = 0;                                         // (the validity words carry the starts)
    // ---- live walk: every unit object starts from init() (prime) or from the state, and goes back there on commit ----
    unsigned long long *grp = L->state + ((size_t)block * A.n_groups + g) * L->group_words;
    unsigned long long *uw = grp + (size_t)warp * W_LIVE_UNIT_WORDS * SYM;
    if (!L->prime) win_live_rings<true>(rings, grp, L->ring_bytes, n_units * 32);
    roles_sync(n_units);                                 // every piece of the ring area is in place
    // the high / low planes' addresses of absolute bar 0 (Ext2's re-reads index them by absolute bar)
    const double *gh = A.in[1] + ((ptrdiff_t)block * L->in_stride - L->t_base) * SYM;
    const double *gl = A.in[2] + ((ptrdiff_t)block * L->in_stride - L->t_base) * SYM;
    auto go = [&](auto &R, auto &&init, auto &&resume) {
        if (L->prime) init();
        else {
            win_live_unit<true>(R, uw, lane);
            resume();
        }
        for (int q = 0; q < (int)(sizeof(R.ovm) / sizeof(R.ovm[0])); ++q) R.ovm[q] = ovm[q];
        __syncwarp();
        run_unit<true, std::remove_reference_t<decltype(R)>, true>(R, A, U, stage, full, cnt, n_units, block, lane, a, L);
        if (L->commit) {
            win_live_unit<false>(R, uw, lane);
            roles_sync(n_units);                         // no unit warp touches the ring area any more
            win_live_rings<false>(rings, grp, L->ring_bytes, n_units * 32);
        }
    };
    auto kdj0 = [&](auto &R) {
        R.fr.init(rings + U.off_fk, U.sk, lane);
        R.sr.init(rings + U.off_sk, U.sd, lane);
        R.s_k = R.s_d = 0.0;
        R.pNum = R.pDen = R.pFk = 0.0;
        R.run_h = R.run_l = R.nfk = R.nsk = 0;
    };
    auto wmd0 = [&](auto &R) { R.pH = R.pL = R.pC = 0.0; R.n_valid = 0; };
    // (bars_padded 0: no copy at init, Ext2T<true>)
    auto two = [&](auto &E) { E.init(rings + U.off_h, unit_p + warp, gh, gl, U.w, U.seg, INT_MAX, lane, src_lane, 0); };
    auto nothing = [] {};
    if (U.kind == WK_KDJ) {
        if (U.off_l >= 0) { UnitKdj<Ext, false> R; go(R, [&] { R.ek.init(rings + U.off_h, rings + U.off_l, U.w, lane); kdj0(R); }, nothing); }
        else { UnitKdj<Ext2T<true>, false> R; go(R, [&] { two(R.ek); kdj0(R); }, [&] { R.ek.resume(unit_p + warp, gh, gl); }); }
    } else if (U.kind == WK_WMD) {
        if (U.off_l >= 0) { UnitWmd<Ext, false> R; go(R, [&] { R.ew.init(rings + U.off_h, rings + U.off_l, U.w, lane); wmd0(R); }, nothing); }
        else { UnitWmd<Ext2T<true>, false> R; go(R, [&] { two(R.ew); wmd0(R); }, [&] { R.ew.resume(unit_p + warp, gh, gl); }); }
    } else {
        UnitAtr R;
        go(R, [&] { R.atr.init(); R.pc = 0.0; R.n_tr = 0; R.pcv = false; }, nothing);
    }
}

}  // namespace pqb
