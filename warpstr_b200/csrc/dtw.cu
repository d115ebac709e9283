// DTW state-automaton fill + traceback for sm_100a.
//
// Replaces WarpSTR._calc_dtw_astates (reference src/caller/caller.py:198-245) and
// WarpSTR._backtracking (:247-301).
//
// One warp owns one read; the automaton's states live in registers, K = KC + KG per lane:
//   * KC "chain" slots: lane l holds KC consecutive states of a pure chain (every state has
//     exactly one incoming edge, from the state before it: the flanks).  Its skip candidate
//     comes from the neighbouring register; slot 0 reads the previous lane's tail.
//   * KG "generic" slots: one arbitrary state per lane and slot (the repeat region: loop
//     back-edges, optional-group skips, IUPAC fan-in, context copies).  Up to DEG incoming
//     edges each, kept in the reference's incoming order, gathered from a small published
//     row in shared memory.
// Row i of the DP needs only row i-1 (stay) and row i-back (skip through an incoming state),
// so per state the warp carries D[i-1] and the running partial sums
//     P_m[t] = D[t] + |x[t+1]-v| + ... + |x[t+m]-v|        m = 1..mv-1
// in the reference's own left-to-right addition order; the skip candidate into state j over
// incoming state p is P_{back-1}[i-back][p] + |x[i]-v_j|, bit-identical to the reference's
// nested loop.  Every row each lane publishes the values other lanes may need (its generic
// states and its chain tail, KG+1 stores), one __syncwarp, then everything is branch-free:
// lanes with fewer edges read a cell that always holds +inf.  All arithmetic is FP64
// add/abs/compare: no multiply, so no FMA contraction can occur.
//
// The read's signal is streamed through shared memory in 1 KB tiles with 1-D bulk async
// copies (cp.async.bulk + mbarrier, TMA engine) two tiles ahead of the row loop.
// Output: a direction code per cell (1 bit for a chain state, DEG bits for a generic one),
// the codes of one lane and 32/NB consecutive rows packed in one 32-bit word, stored
// [word row][lane] so that every word row is one coalesced 128-byte line (see DirFmt).
// D itself never leaves the SM.
#include "wstr_internal.h"

namespace {

constexpr int CH = WSTR_SIG_CHUNK;
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// one elected lane: announce `bytes` and start the bulk copy global -> shared
__device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }

// Per-state registers of one lane.  R holds the mv-1 running partial sums; to avoid moving
// them down the pipeline every row their roles rotate instead: at phase ph the sum P_m lives
// in R[(m - 1 - ph) mod (mv-1)].  A row adds the emission in place to P_1..P_{mv-2} (which
// thereby become P_2..P_{mv-1}) and overwrites the register that held P_{mv-1} with the new
// P_1; mv-1 consecutive rows bring every role back to its register.
template <int K, int MV>
struct LaneState {
    double v[K];
    double D[K];
    double R[MV - 1][K];
};

template <int MV>
__host__ __device__ constexpr int role_reg(int m, int ph) {   // register of P_m at phase ph
    return ((m - 1 - ph) % (MV - 1) + (MV - 1)) % (MV - 1);
}

// the pipeline value a state offers to its successors in this row
template <int K, int MV, bool SHORT, int PH>
__device__ __forceinline__ double offer(const LaneState<K, MV> &s, int k) {
    if (SHORT) {
        if (MV >= 3) return s.R[role_reg<MV>(MV >= 3 ? MV - 2 : 1, PH)][k];
        return s.D[k];
    }
    return s.R[role_reg<MV>(MV - 1, PH)][k];
}

// shift the pipeline of state k by one row: P_m += emission for m < mv-1, P_1 = stay
template <int K, int MV, int PH>
__device__ __forceinline__ void advance(LaneState<K, MV> &s, int k, double ae, double stay) {
#pragma unroll
    for (int m = MV - 2; m >= 1; --m) s.R[role_reg<MV>(m, PH)][k] += ae;
    s.R[role_reg<MV>(MV - 1, PH)][k] = stay;
}

template <int KG>
struct LaneConsts {
    uint32_t band_bits;     // slot u of this lane is inside the end band's skipped prefix
    uint32_t src0;          // byte offset (within a published row) of chain slot 0's predecessor
    uint32_t gsrc[KG];      // generic slot g: 4 x 8-bit published-row indices, incoming order
};

// published row: [generic g][lane] ... [chain tail][lane], [+inf cell]
template <int KG>
__host__ __device__ constexpr int q_row_len() { return 32 * KG + 40; }

// Direction codes.  Per cell a small mask of the candidates that took the lead in turn (bit r =
// incoming edge r, tried in list order, so the winner is the highest set bit; 0 = stay): one
// bit for a chain slot, one bit per candidate of a generic slot, NB bits per lane and row.
// RPW = 32/NB consecutive rows share one 32-bit word per lane (row i: word i/RPW, bit field
// (i%RPW)*NB); a word row [32 lanes] is one coalesced 128-byte line.  HD/FMR1/C9orf72 (6,2,2):
// 10 bits, 3 rows per word = 0.17 B per cell.
// DEG encodes the candidates per generic slot: 2 or 4 = that many for every slot; 100 + d =
// "low" layout, one candidate for every generic slot but the last, d for the last (the host
// puts the states with more than one incoming edge there); 200 + 10 a + b = "graded" layout, a
// candidates for the last slot, b for the one before it, one for the others ((CAN): 21 states with
// four incoming edges, 20 with two, 70 with one -- 8 candidates per lane and row instead of 16).
template <int DEG>
struct DegOf {
    static constexpr bool LOW = DEG >= 100 && DEG < 200;
    static constexpr bool GRADED = DEG >= 200;
    static constexpr int MAX = GRADED ? (DEG - 200) / 10 : (LOW ? DEG - 100 : DEG);
};
template <int KG, int DEG>
__host__ __device__ constexpr int slot_deg(int g) {
    if (DegOf<DEG>::GRADED) return g == KG - 1 ? (DEG - 200) / 10 : (g == KG - 2 ? (DEG - 200) % 10 : 1);
    return (DegOf<DEG>::LOW && g < KG - 1) ? 1 : DegOf<DEG>::MAX;
}
template <int KC, int KG, int DEG>
__host__ __device__ constexpr int slot_bit(int g) {      // first bit of generic slot g in a row's field
    int b = KC;
    for (int i = 0; i < g; ++i) b += slot_deg<KG, DEG>(i);
    return b;
}
template <int KC, int KG, int DEG>
struct DirFmt {
    static constexpr int NB = slot_bit<KC, KG, DEG>(KG - 1) + DegOf<DEG>::MAX;
    static constexpr int RPW = 32 / NB;
    static_assert(NB <= 32 && RPW >= 1, "direction codes of one row must fit a 32-bit word");
};

// running output position of one lane
struct DirOut {
    uint32_t acc;      // bits collected for the current word
    int sh;            // bit offset of the next row inside it
    uint32_t *ptr;     // where the current word goes
};

// min(best, cand) with the reference's strict '<'; when cand wins, OR `bit` into codes.
// (The result is a fresh register on purpose: tying it to `best` would force a copy whenever
// best is still needed, as the stay value is for the pipeline.)
// (Comparing the bit patterns as unsigned integers instead -- legal, every value is a
// non-negative sum or +inf -- moves the compare off the FP64 pipe but costs two to four ISETP
// on the ALU pipe, which the selects and code bits already load: no gain, SASS checked.)
__device__ __forceinline__ double take_min(const double best, uint32_t &codes, const double cand, const uint32_t bit) {
    double out;
    asm("{\n"
        ".reg .pred p;\n"
        "setp.lt.f64 p, %2, %3;\n"
        "selp.f64 %0, %2, %3, p;\n"
        "@p or.b32 %1, %1, %4;\n"
        "}\n"
        : "=d"(out), "+r"(codes)
        : "d"(cand), "d"(best), "r"(bit));
    return out;
}

// One DP row at pipeline phase PH (leaves the state at phase PH+1).
// SHORT: this row allows dwell mv-1 (masked row of the second pass).
// BAND: the end band is active (caller.py:223-224).
// SUB >= 0: the row's position inside its direction word is known at compile time (the word
//   is stored after its last row); SUB < 0: taken from o.sh.
//   Qpub = &Q[lane] of this row's published buffer, Qrow = the buffer itself
template <int KC, int KG, int DEG, int MV, bool SHORT, bool BAND, int PH, int SUB>
__device__ __forceinline__ void dp_row(LaneState<KC + KG, MV> &s, const LaneConsts<KG> &lc, const double x,
                                       double *__restrict__ Qpub, const double *__restrict__ Qrow, DirOut &o) {
    constexpr int K = KC + KG;
    constexpr int NB = DirFmt<KC, KG, DEG>::NB, RPW = DirFmt<KC, KG, DEG>::RPW;
    constexpr int B0 = SUB >= 0 ? SUB * NB : 0;      // bit offset of this row's field in `codes`
    const double INF = dinf();

    // what other lanes may read this row: my generic states and my chain tail
#pragma unroll
    for (int g = 0; g < KG; ++g) Qpub[g * 32] = offer<K, MV, SHORT, PH>(s, KC + g);
    Qpub[KG * 32] = offer<K, MV, SHORT, PH>(s, KC - 1);
    __syncwarp();

    uint32_t codes = SUB >= 0 ? o.acc : 0u;

    // ---- chain slots: stay or the single incoming edge -----------------------------------
    // (last slot first: a slot's candidate is the old pipeline value of the slot below it, which
    // is then still untouched, so every update can happen in place)
    const double qfirst = *reinterpret_cast<const double *>(reinterpret_cast<const unsigned char *>(Qrow) + lc.src0);
#pragma unroll
    for (int k = KC - 1; k >= 0; --k) {
        const double ae = fabs(x - s.v[k]);
        const double qprev = k > 0 ? offer<K, MV, SHORT, PH>(s, k > 0 ? k - 1 : 0) : qfirst;
        const double stay = s.D[k] + ae;
        double best = stay;
        best = take_min(best, codes, qprev + ae, 1u << (B0 + k));
        if (BAND) {
            if ((lc.band_bits >> k) & 1u) {
                best = INF;
                codes &= ~(1u << (B0 + k));
            }
        }
        advance<K, MV, PH>(s, k, ae, stay);
        s.D[k] = best;
    }

    // ---- generic slots: stay, then the slot's incoming edges in list order ------------------------
#pragma unroll
    for (int g = 0; g < KG; ++g) {
        const int k = KC + g;
        const double ae = fabs(x - s.v[k]);
        const double stay = s.D[k] + ae;
        double best = stay;
#pragma unroll
        for (int r = 0; r < DegOf<DEG>::MAX; ++r) {
            if (r < slot_deg<KG, DEG>(g)) {
                const uint32_t idx = (lc.gsrc[g] >> (8 * r)) & 0xffu;
                best = take_min(best, codes, Qrow[idx] + ae, 1u << (B0 + slot_bit<KC, KG, DEG>(g) + r));
            }
        }
        if (BAND) {
            if ((lc.band_bits >> k) & 1u) {
                best = INF;
                codes &= ~(((1u << slot_deg<KG, DEG>(g)) - 1u) << (B0 + slot_bit<KC, KG, DEG>(g)));
            }
        }
        advance<K, MV, PH>(s, k, ae, stay);
        s.D[k] = best;
    }

    if (SUB >= 0) {
        if (SUB == RPW - 1) {
            *o.ptr = codes;
            o.ptr += 32;
            o.acc = 0u;
        } else {
            o.acc = codes;
        }
    } else {
        o.acc |= codes << o.sh;
        o.sh += NB;
        if (o.sh > 32 - NB) {
            *o.ptr = o.acc;
            o.ptr += 32;
            o.acc = 0u;
            o.sh = 0;
        }
    }
}

// mv-1 consecutive rows: every role returns to its register, nothing has to be moved.
// xv holds the rows' samples; each is replaced by the next cycle's as soon as its row is done.
// ALIGNED: the cycle covers exactly one direction word (RPW == mv-1, entered with o.sh == 0).
template <int KC, int KG, int DEG, int MV, bool SHORT, bool BAND, bool ALIGNED, int PH = 0>
__device__ __forceinline__ void dp_rows_cycle(LaneState<KC + KG, MV> &s, const LaneConsts<KG> &lc,
                                              double (&xv)[MV - 1], const double *__restrict__ xnext,
                                              double *__restrict__ Qlane, const double *__restrict__ Qbase,
                                              DirOut &o) {
    constexpr int QL = q_row_len<KG>();
    constexpr int RPW = DirFmt<KC, KG, DEG>::RPW;
    constexpr int SUB = RPW == 1 ? 0 : (ALIGNED ? PH : -1);
    dp_row<KC, KG, DEG, MV, SHORT, BAND, PH, SUB>(s, lc, xv[PH], Qlane + PH * QL, Qbase + PH * QL, o);
    xv[PH] = xnext[PH];   // the same phase's sample of the next cycle, a whole cycle ahead of its use
    if constexpr (PH + 1 < MV - 1)
        dp_rows_cycle<KC, KG, DEG, MV, SHORT, BAND, ALIGNED, PH + 1>(s, lc, xv, xnext, Qlane, Qbase, o);
}

// a single row from phase 0 back to phase 0 (registers rotated by hand; used for the few rows
// that do not fill a cycle)
template <int KC, int KG, int DEG, int MV, bool SHORT, bool BAND>
__device__ __forceinline__ void dp_row_single(LaneState<KC + KG, MV> &s, const LaneConsts<KG> &lc, const double x,
                                              double *__restrict__ Qlane, const double *__restrict__ Qbase,
                                              DirOut &o) {
    constexpr int K = KC + KG;
    constexpr int SUB = DirFmt<KC, KG, DEG>::RPW == 1 ? 0 : -1;
    dp_row<KC, KG, DEG, MV, SHORT, BAND, 0, SUB>(s, lc, x, Qlane, Qbase, o);
    __syncwarp();   // the next row publishes into the same buffer
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const double last = s.R[MV - 2][k];
#pragma unroll
        for (int m = MV - 2; m >= 1; --m) s.R[m][k] = s.R[m - 1][k];
        s.R[0][k] = last;
    }
}

// rows [i0, i1) of the tile starting at row `tile0`, one (SHORT, BAND) setting
template <int KC, int KG, int DEG, int MV, bool SHORT, bool BAND>
__device__ __forceinline__ void dp_segment(LaneState<KC + KG, MV> &s, const LaneConsts<KG> &lc,
                                           const double *__restrict__ xs, const int tile0, int i0, const int i1,
                                           double *__restrict__ Qlane, const double *__restrict__ Qbase, DirOut &o) {
    constexpr int CY = MV - 1;
    constexpr int RPW = DirFmt<KC, KG, DEG>::RPW;
    constexpr bool ALIGNED = RPW == CY && RPW > 1;
    const double *xp = xs + (i0 - tile0);
    if (ALIGNED) {   // single rows up to the next word boundary, so that every cycle fills one word
#pragma unroll 1
        for (; i0 < i1 && o.sh != 0; ++i0) {
            dp_row_single<KC, KG, DEG, MV, SHORT, BAND>(s, lc, *xp, Qlane, Qbase, o);
            xp += 1;
        }
    }
    double xv[CY];
#pragma unroll
    for (int j = 0; j < CY; ++j) xv[j] = xp[j];          // may run a few samples past the tile: unused then
#pragma unroll 1
    for (; i0 + CY <= i1; i0 += CY) {
        dp_rows_cycle<KC, KG, DEG, MV, SHORT, BAND, ALIGNED>(s, lc, xv, xp + CY, Qlane, Qbase, o);
        xp += CY;
    }
#pragma unroll 1
    for (; i0 < i1; ++i0) {
        dp_row_single<KC, KG, DEG, MV, SHORT, BAND>(s, lc, *xp, Qlane, Qbase, o);
        xp += 1;
    }
}

// first row in (a, limit] whose mask bit differs from row a's (or limit)
__device__ __forceinline__ int mask_run_end(const uint32_t *__restrict__ mw, int a, const int limit, uint32_t &bit) {
    uint32_t word = __ldg(mw + (a >> 5));
    bit = (word >> (a & 31)) & 1u;
    uint32_t diff = (bit ? ~word : word) >> (a & 31);
    int b = a;
    for (;;) {
        if (diff) {
            b += __ffs(diff) - 1;
            break;
        }
        b = (b | 31) + 1;                // next word
        if (b >= limit) break;
        word = __ldg(mw + (b >> 5));
        diff = bit ? ~word : word;
    }
    return b < limit ? b : limit;
}

// rows [i0, i1) of one signal tile (all inside one band setting); mask bits pick SHORT rows
template <int KC, int KG, int DEG, int MV, bool BAND, bool MASKED>
__device__ __forceinline__ void dp_tile_rows(LaneState<KC + KG, MV> &s, const LaneConsts<KG> &lc,
                                             const double *__restrict__ xs, const int tile0, int i0, const int i1,
                                             const uint32_t *__restrict__ mw_ptr, double *__restrict__ Qlane,
                                             const double *__restrict__ Qbase, DirOut &o) {
    if (!MASKED || !mw_ptr) {
        dp_segment<KC, KG, DEG, MV, false, BAND>(s, lc, xs, tile0, i0, i1, Qlane, Qbase, o);
        return;
    }
    while (i0 < i1) {
        uint32_t bit;
        const int b = mask_run_end(mw_ptr, i0, i1, bit);
        if (bit) dp_segment<KC, KG, DEG, MV, true, BAND>(s, lc, xs, tile0, i0, b, Qlane, Qbase, o);
        else dp_segment<KC, KG, DEG, MV, false, BAND>(s, lc, xs, tile0, i0, b, Qlane, Qbase, o);
        i0 = b;
    }
}

// ------------------------------------------------------------------------------------------
// Traceback: follow the stored direction codes from (T-1, endstate) to row 0.  The
// reference re-derives each step by recomputing the candidates and picking the one that
// reproduces the stored cost (caller.py:254-299); the winner of the fill reproduces it
// exactly, so following the fill's arg-min with the same priority (stay, then incoming in
// list order) visits the same cells.
//
// Done by the warp that filled the read, right after the fill.  The direction words are
// staged through shared memory in windows of WRW word rows (one bulk async copy each, a ring
// of NBUF windows in flight), so the walk never waits on HBM for a dependent step.  Inside a window lane t looks at row hi-t: every lane extracts the code
// of the path's current state in its own row, one ballot finds the first row that is not a
// "stay", all rows above it are emitted at once, and only the state changes (one per ~9
// samples) cost a dependent step.  The trace is written one window at a time.
// ------------------------------------------------------------------------------------------
template <int RPW>
struct TbGeom {
    static constexpr int WRW = RPW == 1 ? 16 : 32 / RPW;   // word rows per window (<= 32 DP rows)
    static constexpr int ROWS = WRW * RPW;                 // DP rows per window
    static constexpr int NBUF = 5;                         // windows in flight
    static constexpr int WORDS = NBUF * WRW * 32;
};

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
template <int KC, int KG, int DEG>
__device__ __forceinline__ void traceback_warp(const DevAutomaton *A, const int T, const uint32_t *dir,
                                               const uint32_t *mw, int32_t *tr, int32_t *status_slot,
                                               const int lane, uint32_t *win, uint64_t *bar, uint32_t &phase_bits,
                                               const int32_t *spred) {
    constexpr int K = KC + KG;
    constexpr int NB = DirFmt<KC, KG, DEG>::NB, RPW = DirFmt<KC, KG, DEG>::RPW;
    using G = TbGeom<RPW>;
    constexpr int WRW = G::WRW, ROWS = G::ROWS, NBUF = G::NBUF;
    const int mv = A->mv;
    const int wtop = (T - 1) / RPW;                  // last word row
    const int wmin = mv / RPW;                       // first word row that was written
    const int nwin = wtop / WRW + 1;

    // window c holds word rows wh-WRW+1 .. wh (wh = wtop - c*WRW) in memory order: one bulk copy
    auto issue = [&](int c) {
        if (lane != 0) return;
        const int b = c % NBUF;
        const int wh = wtop - c * WRW;
        const int wfirst = wh - WRW + 1;
        const int w0 = wfirst > wmin ? wfirst : wmin;      // word rows below wmin were never written
        const int n = wh - w0 + 1;
        if (n > 0)
            bulk_load(win + (b * WRW + (w0 - wfirst)) * 32, dir + static_cast<int64_t>(w0) * 32,
                      static_cast<uint32_t>(n) * 128u, &bar[b]);
        else
            mbar_expect_tx(&bar[b], 0u);
    };

    int i = T - 1;
    int pos = A->end_pos;
    int st = __ldg(A->state_of_pos + pos);
    bool failed = false;
    for (int c = 0; c < nwin && c < NBUF; ++c) issue(c);

    for (int c = 0; c < nwin; ++c) {
        const int b = c % NBUF;
        while (!mbar_try_wait(&bar[b], (phase_bits >> b) & 1u)) {
        }
        phase_bits ^= 1u << b;
        const int wh = wtop - c * WRW;
        const int hi = wh * RPW + RPW - 1;            // may lie past T-1 in the first window
        const int lo = hi - ROWS + 1 > 0 ? hi - ROWS + 1 : 0;
        if (i >= lo && i > 0 && !failed) {
            const int row = hi - lane;
            // rows of this window the walk enters from above (rows above i were emitted with the
            // previous window's last move)
            const bool mine = lane < ROWS && row >= lo && row <= i;
            const bool coded = mine && row >= mv;
            uint32_t mb = 0u;
            if (mw && mine) mb = (__ldg(mw + (row >> 5)) >> (row & 31)) & 1u;
            const int wr = mine ? row / RPW : wh;
            const uint32_t *wslot = win + (b * WRW + (wr - (wh - WRW + 1))) * 32;
            const int fsh = (row - wr * RPW) * NB;      // this row's bit field inside its word
            int my = st;                                // state emitted for this lane's row
            for (;;) {
                const int hl = pos / K;
                const int u = pos - hl * K;
                // code of the path's state in this lane's row (0 = stay)
                uint32_t nib = 0u;
                if (coded && row <= i) {
                    const uint32_t f = wslot[hl] >> fsh;
                    if (u < KC) {
                        nib = (f >> u) & 1u;
                    } else {
                        const int g = u - KC;
                        int off = KC, width = 1;
#pragma unroll
                        for (int gg = 0; gg < KG; ++gg)
                            if (g == gg) {
                                off = slot_bit<KC, KG, DEG>(gg);
                                width = slot_deg<KG, DEG>(gg);
                            }
                        nib = (f >> off) & ((1u << width) - 1u);
                    }
                }
                const uint32_t moves = __ballot_sync(FULL, nib != 0u);
                if (moves == 0u) {                          // stays down to the window's last row
                    i = lo - 1;
                    break;
                }
                const int tm = __ffs(moves) - 1;            // lane of the first row that leaves the state
                const int rm = hi - tm;
                const uint32_t nibm = __shfl_sync(FULL, nib, tm);
                const int back = mv - static_cast<int>(__shfl_sync(FULL, mb, tm));
                const int code = 31 - __clz(nibm);          // last candidate that took the lead
                const int32_t pp = spred[pos * DegOf<DEG>::MAX + code];
                if (rm < back || pp < 0) {
                    failed = true;
                    break;
                }
                const int pst = pp >> 16;
                // the move row keeps the state it leaves; every row below it belongs to the
                // predecessor until a later move says otherwise
                if (row < rm) my = pst;
                if (rm - back + 1 < lo) {                   // skipped rows below this window
                    const int r = lo - 1 - lane;
                    if (lane < back - 1 && r > rm - back) tr[r] = pst;
                }
                i = rm - back;
                pos = pp & 0xffff;
                st = pst;
                if (i < lo || i <= 0) break;
            }
            if (mine) tr[row] = my;
        }
        __syncwarp();                                       // every lane is done with this buffer
        if (c + NBUF < nwin) issue(c + NBUF);
    }
    if (lane == 0) {
        if (failed) *status_slot = WSTR_READ_BACKTRACK;
        else tr[0] = st;
    }
}

// per-warp shared memory
template <int KC, int KG, int DEG, int MV>
struct alignas(16) FillSmem {
    using G = TbGeom<DirFmt<KC, KG, DEG>::RPW>;
    double sig[2][CH];                   // look-ahead reads may run up to 2*(mv-1) samples past a tile (into Q: unused)
    double Q[MV - 1][q_row_len<KG>()];   // one published buffer per pipeline phase
    uint32_t win[G::WORDS];              // traceback windows
    int32_t pred[(KC + KG) * 32 * DegOf<DEG>::MAX];  // traceback: (state << 16 | position) of the predecessor, by position and code
    uint64_t bar[2];                     // signal tiles
    uint64_t tbar[G::NBUF];              // traceback windows
};

// Resident warps per SM the register budget is set for, by states per lane.  Warps are bound to
// one of the SM's four sub-partitions (16 K registers each): 12 warps = 3 per sub-partition =
// 168 registers per thread, 13..16 warps = 4 per sub-partition = 128.  With one-warp CTAs the
// (7,1) and (8,1) row loops fit 128 registers (no spill in the first-pass loop, one or two local
// loads per 3-row cycle in the masked second-pass variants), and 16 warps are 2 % faster than 12.
// The per-lane state is (KC+KG)*(MV+1) doubles; beyond 45 of them (min_values_per_state 5 or 6) the
// loops would spill at 128 registers, so those keep the 12-warp budget; so do the layouts with two or more
// generic slots (their candidates' addresses and values do not fit next to nine states); beyond 60 doubles of
// state (long dwells on wide layouts) 8 warps and 255 registers.  The MASKED
// instantiation (second pass: rows whose mask bit is set allow the shorter dwell): its extra row
// variants spill a few values per cycle at 128 registers, which costs what the fourth warp gains
// (41.7 ms per pass either way).  The first-pass instantiation does not contain the masked variants
// at all and has no local-memory access in its row loop.
#ifndef WSTR_K8_WARPS
#define WSTR_K8_WARPS 16
#endif
#ifdef WSTR_MAXNREG
#define WSTR_FILL_BOUNDS __maxnreg__(WSTR_MAXNREG)
#else
#define WSTR_FILL_BOUNDS                         \
    __launch_bounds__(32 * WSTR_WARPS_PER_CTA,   \
                      ((KC + KG) * (MV + 1) <= 45 && KG <= 1 && !MASKED ? WSTR_K8_WARPS                                          \
                       : ((KC + KG) * (MV + 1) <= 60 && KC + KG <= 12 ? 12 : 8)) / WSTR_WARPS_PER_CTA)
#endif
template <int KC, int KG, int DEG, int MV, bool MASKED>
__global__ void WSTR_FILL_BOUNDS dtw_fill_kernel(const FillParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int K = KC + KG;
    constexpr int NB = DirFmt<KC, KG, DEG>::NB, RPW = DirFmt<KC, KG, DEG>::RPW;
    // (one-warp CTAs: say so outright, so that every shared-memory address below is a constant)
    const int warp = WSTR_WARPS_PER_CTA == 1 ? 0 : static_cast<int>(threadIdx.x >> 5);
    const int lane = WSTR_WARPS_PER_CTA == 1 ? static_cast<int>(threadIdx.x) : static_cast<int>(threadIdx.x & 31);
    using Smem = FillSmem<KC, KG, DEG, MV>;
    Smem &sm = reinterpret_cast<Smem *>(smem_raw)[warp];
    const double INF = dinf();

    if (lane == 0) {
        mbar_init(&sm.bar[0], 1);
        mbar_init(&sm.bar[1], 1);
        for (int b = 0; b < Smem::G::NBUF; ++b) mbar_init(&sm.tbar[b], 1);
        fence_barrier_init();
    }
    for (int e = lane; e < (MV - 1) * q_row_len<KG>(); e += 32) (&sm.Q[0][0])[e] = INF;   // incl. the +inf cell
    __syncwarp();
    uint32_t uses0 = 0, uses1 = 0;   // completed phases of the two tile barriers
    uint32_t tb_phase = 0;           // parity bits of the traceback window barriers

    LaneState<K, MV> s;
    LaneConsts<KG> lc;
    int cached_aut = -1;
    double v0 = 0.0;

    // (a counted loop on purpose -- no warp can take more than p.n reads: with `for (;;)` ptxas emits
    // the row loops a third longer, 297 instead of 262 instructions per 3-row cycle, and does not
    // fold the shared-memory addresses; checked in the SASS)
    for (int taken = 0; taken < p.n; ++taken) {
        int r = 0;
        if (lane == 0) r = atomicAdd(p.queue, 1);
        r = __shfl_sync(FULL, r, 0);
        if (r >= p.n) break;
        const ReadMeta m = p.meta[p.order[r]];
        const DevAutomaton *A = p.auts + m.aut;
        const int T = m.T;
        if (p.respect_status && p.status[m.read] != WSTR_READ_OK) continue;   // failed earlier in the call
        if (T <= MV) {
            if (lane == 0) p.status[m.read] = WSTR_READ_TOO_SHORT;
            continue;
        }

        if (m.aut != cached_aut) {   // (re)load the automaton into registers
#pragma unroll
            for (int k = 0; k < K; ++k) s.v[k] = __ldg(A->v_pos + lane * K + k);
            lc.band_bits = __ldg(A->lane_tab + lane * WSTR_LANE_TAB_STRIDE + 0);
            lc.src0 = __ldg(A->lane_tab + lane * WSTR_LANE_TAB_STRIDE + 1) * 8u;
#pragma unroll
            for (int g = 0; g < KG; ++g) lc.gsrc[g] = __ldg(A->lane_tab + lane * WSTR_LANE_TAB_STRIDE + 2 + g);
            v0 = __ldg(A->v_pos + A->init_pos[0]);
            constexpr int DM = DegOf<DEG>::MAX;
            for (int e = lane; e < K * 32 * DM; e += 32)
                sm.pred[e] = __ldg(A->pred_tab + (e / DM) * WSTR_PRED_STRIDE + 1 + (e % DM));
            cached_aut = m.aut;
        }

        // ---- signal tiles: two in flight --------------------------------------------------
        const double *gsig = p.signal + m.sig_off;
        const int nchunks = (T + CH - 1) / CH;
        auto issue = [&](int c) {
            if (lane == 0) {
                int n = T - c * CH;
                n = n > CH ? CH : n;
                n = (n + 1) & ~1;   // 16-byte granules
                bulk_load(sm.sig[c & 1], gsig + static_cast<int64_t>(c) * CH, static_cast<uint32_t>(n) * 8u,
                          &sm.bar[c & 1]);
            }
        };
        issue(0);
        if (nchunks > 1) issue(1);
        while (!mbar_try_wait(&sm.bar[0], uses0 & 1u)) {
        }
        ++uses0;

        // ---- row 0 (caller.py:201-208) and the empty rows 1..mv-1 -----------------------
        {
            const double *x0 = sm.sig[0];
            const double first = fabs(x0[0] - v0);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                s.D[k] = INF;
#pragma unroll
                for (int mm = 0; mm < MV - 1; ++mm) s.R[mm][k] = INF;
            }
            for (int c = 0; c <= MV; ++c) {
                const int pos = A->init_pos[c];
                double d0 = first;
                if (c > 0) d0 = first + fabs(x0[c] - v0);   // row 0, column c
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    if (pos == lane * K + k) {
                        double acc = d0;
                        for (int t = 1; t <= MV - 1; ++t) acc = acc + fabs(x0[t] - s.v[k]);
                        s.R[MV - 2][k] = acc;   // P_{mv-1}[0] (phase 0)
                    }
                }
            }
        }

        const int band_start = max(A->th1, T - A->band6 + 1);
        // mv rows into the band every value computed before it has left the pipelines; if no edge
        // enters the skipped set from outside, its cells then stay +inf (and their codes 0) without
        // the per-cell test
        const int band_free = A->band_closed ? band_start + MV : T;
        const uint32_t *mw_ptr = MASKED && p.maskbits ? p.maskbits + m.mask_off : nullptr;
        uint32_t *dir = p.dir + m.dir_off;
        DirOut o;   // rows below mv leave their bits 0
        o.acc = 0u;
        o.sh = (MV % RPW) * NB;
        o.ptr = dir + (MV / RPW) * 32 + lane;
        double *Qlane = &sm.Q[0][0] + lane;
        const double *Qbase = &sm.Q[0][0];

        for (int c = 0; c < nchunks; ++c) {
            if (c > 0) {
                if (c & 1) {
                    while (!mbar_try_wait(&sm.bar[1], uses1 & 1u)) {
                    }
                    ++uses1;
                } else {
                    while (!mbar_try_wait(&sm.bar[0], uses0 & 1u)) {
                    }
                    ++uses0;
                }
            }
            const double *xs = sm.sig[c & 1];
            const int i_begin = c == 0 ? MV : c * CH;
            const int i_end = min(T, (c + 1) * CH);
            // rows [band_start, band_free) carry the end band's per-cell test, the others do not
            for (int a = i_begin; a < i_end;) {
                const bool banded = a >= band_start && a < band_free;
                const int e = banded ? min(i_end, band_free) : (a < band_start ? min(i_end, band_start) : i_end);
                if (banded) dp_tile_rows<KC, KG, DEG, MV, true, MASKED>(s, lc, xs, c * CH, a, e, mw_ptr, Qlane, Qbase, o);
                else dp_tile_rows<KC, KG, DEG, MV, false, MASKED>(s, lc, xs, c * CH, a, e, mw_ptr, Qlane, Qbase, o);
                a = e;
            }
            __syncwarp();                          // every lane is done with this tile
            if (c + 2 < nchunks) issue(c + 2);     // refill it
        }

        if (o.sh != 0) *o.ptr = o.acc;   // the last, partly filled word
        if (p.end_cost) {
            const int ep = A->end_pos;
#pragma unroll
            for (int k = 0; k < K; ++k)
                if (ep == lane * K + k) p.end_cost[m.read] = s.D[k];
        }
        if (lane == 0) p.status[m.read] = WSTR_READ_OK;
        __syncwarp();   // this warp's direction words are visible to all of its lanes
#ifndef WSTR_NO_TRACEBACK   // (experiment switch: time the fill alone)
        traceback_warp<KC, KG, DEG>(A, T, dir, mw_ptr, p.trace + m.sig_off, p.status + m.read, lane, sm.win, sm.tbar,
                                    tb_phase, sm.pred);
#endif
    }
}

template <int KC, int KG, int DEG, int MV, bool MASKED>
int launch_fill_m(const FillParams &p, cudaStream_t s) {
    static int grid_cap = 0;
    static unsigned long long attr_done = 0ull;      // devices (by ordinal) the function attributes are set on
    const int smem = static_cast<int>(sizeof(FillSmem<KC, KG, DEG, MV>)) * WSTR_WARPS_PER_CTA;
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    if (grid_cap == 0 || !((attr_done >> (dev & 63)) & 1ull)) {
        WSTR_CUDA(cudaFuncSetAttribute(dtw_fill_kernel<KC, KG, DEG, MV, MASKED>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        // (shared memory must not be what limits the resident warps: take the largest carve-out)
        WSTR_CUDA(cudaFuncSetAttribute(dtw_fill_kernel<KC, KG, DEG, MV, MASKED>,
                                       cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
        int sms = 0, per_sm = 0;
        WSTR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        WSTR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dtw_fill_kernel<KC, KG, DEG, MV, MASKED>,
                                                                32 * WSTR_WARPS_PER_CTA, smem));
        if (per_sm < 1) per_sm = 1;
        grid_cap = sms * per_sm;
        attr_done |= 1ull << (dev & 63);
    }
    int grid = (p.n + WSTR_WARPS_PER_CTA - 1) / WSTR_WARPS_PER_CTA;
    if (grid > grid_cap) grid = grid_cap;
    if (grid < 1) return WSTR_OK;
    dtw_fill_kernel<KC, KG, DEG, MV, MASKED><<<grid, 32 * WSTR_WARPS_PER_CTA, smem, s>>>(p);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}

// first pass (no mask) and second pass (mask bits) are separate instantiations, see WSTR_FILL_BOUNDS
template <int KC, int KG, int DEG, int MV>
int launch_fill_t(const FillParams &p, cudaStream_t s) {
    if (p.maskbits) return launch_fill_m<KC, KG, DEG, MV, true>(p, s);
    return launch_fill_m<KC, KG, DEG, MV, false>(p, s);
}

template <int KC, int KG, int MV>
int launch_fill_deg(int deg, const FillParams &p, cudaStream_t s) {
    if (deg == 2) return launch_fill_t<KC, KG, 2, MV>(p, s);
    if (deg == 4) return launch_fill_t<KC, KG, 4, MV>(p, s);
    if constexpr (KG >= 2 && MV == 4) {     // low layouts: one candidate for all generic slots but the last
        if (deg == 102) return launch_fill_t<KC, KG, 102, MV>(p, s);
        if (deg == 104) return launch_fill_t<KC, KG, 104, MV>(p, s);
    }
    if constexpr (KG >= 3 && MV == 4) {     // graded layout: 4 candidates for the last slot, 2 for the one before
        if (deg == 242) return launch_fill_t<KC, KG, 242, MV>(p, s);
    }
    return WSTR_ERR_UNSUPPORTED;
}

}  // namespace

// The (chain, generic) slot splits the library is built with: the same as kSplits in api.cu
// (tests/test_fill_dispatch.py checks both lists and that every instantiation has a test target).
// The instantiations take minutes to compile, so this file is compiled several times in parallel, each
// time with -DWSTR_FILL_PART=n for one group of them (__graft_entry__.py: FILL_PARTS); without the macro
// everything lands in one object.
#ifdef WSTR_FILL_PART
#define WSTR_HAS_PART(n) (WSTR_FILL_PART == (n))
#else
#define WSTR_HAS_PART(n) 1
#endif
#define WSTR_CASE(KC_, KG_, MV_) \
    if (kc == KC_ && kg == KG_ && mv == MV_) return launch_fill_deg<KC_, KG_, MV_>(deg, p, s);

#define WSTR_DECL_PART(n) int wstr_launch_fill_p##n(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s);
WSTR_DECL_PART(0)
WSTR_DECL_PART(1)
WSTR_DECL_PART(2)
WSTR_DECL_PART(3)
WSTR_DECL_PART(4)
WSTR_DECL_PART(5)
WSTR_DECL_PART(6)
WSTR_DECL_PART(7)
WSTR_DECL_PART(8)
#undef WSTR_DECL_PART

#if WSTR_HAS_PART(0)
int wstr_launch_fill_p0(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(7, 1, 4)
    WSTR_CASE(8, 1, 4)
    WSTR_CASE(6, 2, 2)
    WSTR_CASE(6, 2, 3)
    return WSTR_ERR_UNSUPPORTED;
}

int wstr_launch_fill(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    typedef int (*part_fn)(int, int, int, int, const FillParams &, cudaStream_t);
    static const part_fn parts[] = {wstr_launch_fill_p0, wstr_launch_fill_p1, wstr_launch_fill_p2,
                                    wstr_launch_fill_p3, wstr_launch_fill_p4, wstr_launch_fill_p5,
                                    wstr_launch_fill_p6, wstr_launch_fill_p7, wstr_launch_fill_p8};
    for (part_fn f : parts) {
        const int rc = f(kc, kg, deg, mv, p, s);
        if (rc != WSTR_ERR_UNSUPPORTED) return rc;
    }
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#if WSTR_HAS_PART(1)
int wstr_launch_fill_p1(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(6, 2, 4)
    WSTR_CASE(6, 2, 5)
    WSTR_CASE(6, 2, 6)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#if WSTR_HAS_PART(2)
int wstr_launch_fill_p2(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(4, 4, 4)
    WSTR_CASE(8, 2, 4)
    WSTR_CASE(6, 4, 4)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#if WSTR_HAS_PART(3)
int wstr_launch_fill_p3(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(8, 4, 4)
    WSTR_CASE(12, 4, 4)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
// (6,4) holds every automaton of up to ~320 states: the specialised kernel of the other dwell settings
#if WSTR_HAS_PART(4)
int wstr_launch_fill_p4(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(6, 4, 2)
    WSTR_CASE(6, 4, 3)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#if WSTR_HAS_PART(5)
int wstr_launch_fill_p5(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(6, 4, 5)
    WSTR_CASE(6, 4, 6)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
// nine and eleven states per lane: DM2 / RFC1 (265-267 states) and the 324-state strand of (CAN) without
// the padding of the (8,2) and (8,4) splits
#if WSTR_HAS_PART(6)
int wstr_launch_fill_p6(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(7, 2, 4)
    WSTR_CASE(7, 4, 4)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
// long dwells (min_values_per_state 7, 8: seven or eight running sums per state, 8 warps per SM)
#if WSTR_HAS_PART(7)
int wstr_launch_fill_p7(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(6, 2, 7)
    WSTR_CASE(6, 2, 8)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#if WSTR_HAS_PART(8)
int wstr_launch_fill_p8(int kc, int kg, int deg, int mv, const FillParams &p, cudaStream_t s) {
    WSTR_CASE(6, 4, 7)
    WSTR_CASE(6, 4, 8)
    return WSTR_ERR_UNSUPPORTED;
}
#endif
#undef WSTR_CASE
