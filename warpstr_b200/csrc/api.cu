// Host side of the C ABI: automaton layout + upload, wave scheduling of the DP passes.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <numeric>
#include <vector>

#include "wstr_internal.h"

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_cuda_err[512] = "";

int wstr_set_cuda_error(cudaError_t e, const char *where) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return WSTR_ERR_NO_DEVICE;
    return WSTR_ERR_CUDA;
}

extern "C" int wstr_version(void) { return 100; }

extern "C" const char *wstr_last_cuda_error(void) { return g_cuda_err; }

extern "C" const char *wstr_error_string(int code) {
    switch (code) {
        case WSTR_OK: return "ok";
        case WSTR_ERR_INVALID_ARGUMENT: return "invalid argument";
        case WSTR_ERR_CUDA: return "CUDA error (see wstr_last_cuda_error)";
        case WSTR_ERR_TOO_MANY_STATES:
            return "automaton too large: states x min_values_per_state exceeds the catch-all kernel's shared memory";
        case WSTR_ERR_UNSUPPORTED: return "unsupported configuration";
        case WSTR_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
        case WSTR_ERR_NO_DEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}

// ------------------------------------------------------------------------------------------
// kernel timing (CUDA events on the launching stream)
// ------------------------------------------------------------------------------------------
namespace {
struct ProfSpan {
    int cat;
    cudaEvent_t a, b;
};
bool g_prof_on = false;
std::vector<ProfSpan> g_prof_spans;
}  // namespace

void wstr_prof_begin(int cat, cudaStream_t s) {
    if (!g_prof_on) return;
    ProfSpan sp;
    sp.cat = cat;
    cudaEventCreate(&sp.a);
    cudaEventCreate(&sp.b);
    cudaEventRecord(sp.a, s);
    g_prof_spans.push_back(sp);
}

void wstr_prof_end(cudaStream_t s) {
    if (!g_prof_on || g_prof_spans.empty()) return;
    cudaEventRecord(g_prof_spans.back().b, s);
}

extern "C" int wstr_profile_enable(int32_t on) {
    g_prof_on = on != 0;
    return WSTR_OK;
}

extern "C" int wstr_profile_read(double *ms, int32_t *launches, int32_t n) {
    if (!ms || !launches || n <= 0) return WSTR_ERR_INVALID_ARGUMENT;
    for (int i = 0; i < n; ++i) {
        ms[i] = 0.0;
        launches[i] = 0;
    }
    for (ProfSpan &sp : g_prof_spans) {
        cudaError_t e = cudaEventSynchronize(sp.b);
        float t = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&t, sp.a, sp.b);
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
        if (e != cudaSuccess) {
            g_prof_spans.clear();
            return wstr_set_cuda_error(e, "wstr_profile_read");
        }
        if (sp.cat >= 0 && sp.cat < n) {
            ms[sp.cat] += t;
            launches[sp.cat] += 1;
        }
    }
    g_prof_spans.clear();
    return WSTR_OK;
}

// ------------------------------------------------------------------------------------------
// automaton layout (see dtw.cu)
//
// A "chain link" j -> t is an edge where j has no other successor and t no other predecessor.
// Maximal chains of links (the flanks, mostly) are cut into full lanes of KC states, taken
// from the chain's end so that the last state of every chain is a lane tail (published);
// everything else (chain heads that do not fill a lane, the repeat region) becomes a
// generic state.  Among the (KC, KG) splits the library is built with, the cheapest one
// that fits is used.
// ------------------------------------------------------------------------------------------
namespace {

bool g_generic_only = false;   // wstr_set_generic_only: build automata for the catch-all kernel only

struct Split {
    int kc, kg;
    unsigned mv_mask;   // bit mv set = instantiated for that min_values_per_state
};
// the same splits as the WSTR_CASE lines of wstr_launch_fill in dtw.cu (tests/test_fill_dispatch.py checks it)
const Split kSplits[] = {{7, 1, 0x10}, {6, 2, 0x1fc}, {8, 1, 0x10}, {4, 4, 0x10}, {7, 2, 0x10}, {8, 2, 0x10},
                         {6, 4, 0x1fc}, {7, 4, 0x10}, {8, 4, 0x10}, {12, 4, 0x10}};

struct Layout {
    int KC = 0, KG = 0, DEG = 2, n_lanes = 0, n_generic = 0;
    std::vector<int> state_of_pos;   // 32*K, -1 padding
    std::vector<int> pos_of_state;   // S
};

struct Chains {
    std::vector<std::vector<int>> seqs;   // maximal chains (>= 1 state each), every state in exactly one
    std::vector<int> indeg, outdeg;
};

Chains find_chains(int S, const int32_t *in_ptr, const int32_t *in_idx) {
    Chains c;
    c.indeg.assign(S, 0);
    c.outdeg.assign(S, 0);
    for (int j = 0; j < S; ++j) {
        c.indeg[j] = in_ptr[j + 1] - in_ptr[j];
        for (int e = in_ptr[j]; e < in_ptr[j + 1]; ++e) c.outdeg[in_idx[e]]++;
    }
    std::vector<int> link_next(S, -1), link_prev(S, -1);
    for (int t = 0; t < S; ++t) {
        if (c.indeg[t] != 1) continue;
        const int j = in_idx[in_ptr[t]];
        if (j == t || c.outdeg[j] != 1) continue;
        link_next[j] = t;
        link_prev[t] = j;
    }
    std::vector<char> seen(S, 0);
    for (int h = 0; h < S; ++h) {
        if (link_prev[h] != -1) continue;
        std::vector<int> seq;
        for (int j = h; j != -1 && !seen[j]; j = link_next[j]) {
            seen[j] = 1;
            seq.push_back(j);
        }
        c.seqs.push_back(seq);
    }
    for (int h = 0; h < S; ++h)   // pure cycles of links (unreachable in practice)
        if (!seen[h]) {
            std::vector<int> seq;
            for (int j = h; !seen[j]; j = link_next[j]) {
                seen[j] = 1;
                seq.push_back(j);
            }
            // break the cycle: its first state is treated as a head with a (published) predecessor
            c.seqs.push_back(seq);
        }
    return c;
}

// lanes each chain gets under a given KC; returns total lanes
int plan_lanes(const Chains &c, int KC, std::vector<int> &lanes) {
    lanes.assign(c.seqs.size(), 0);
    int total = 0;
    for (size_t i = 0; i < c.seqs.size(); ++i) {
        const std::vector<int> &q = c.seqs[i];
        int eligible = (int)q.size();
        if (c.indeg[q[0]] > 1) eligible -= 1;           // a merge point can only be generic
        if (c.indeg[q[0]] == 1 && (int)q.size() > 0) {
            // head with one predecessor: fine as slot 0 as long as that predecessor is published,
            // which holds because the predecessor ends its own chain (it is not linked to us)
        }
        lanes[i] = eligible / KC;
        total += lanes[i];
    }
    while (total > 32) {   // give lanes back, shortest surplus first: take from the longest chain
        size_t best = 0;
        for (size_t i = 1; i < lanes.size(); ++i)
            if (lanes[i] > lanes[best]) best = i;
        lanes[best]--;
        total--;
    }
    return total;
}

int build_layout(int S, const int32_t *in_ptr, const int32_t *in_idx, int mv, Layout &L) {
    const Chains c = find_chains(S, in_ptr, in_idx);
    int best_cost = 1 << 30, best_split = -1;
    std::vector<int> lanes, best_lanes;
    int max_indeg_all = 0;
    for (int j = 0; j < S; ++j) max_indeg_all = std::max(max_indeg_all, c.indeg[j]);
    for (size_t si = 0; si < sizeof(kSplits) / sizeof(kSplits[0]); ++si) {
        const Split &sp = kSplits[si];
        if (!((sp.mv_mask >> mv) & 1u)) continue;
        const int total = plan_lanes(c, sp.kc, lanes);
        const int generic = S - total * sp.kc;
        if (generic > 32 * sp.kg) continue;
        const int deg = max_indeg_all <= 2 ? 2 : 4;
        const int cost = sp.kc * 9 + sp.kg * (8 + 8 * deg);
        if (cost < best_cost) {
            best_cost = cost;
            best_split = (int)si;
            best_lanes = lanes;
        }
    }
    if (best_split < 0) {
        bool any_mv = false;
        for (const Split &sp : kSplits) any_mv |= ((sp.mv_mask >> mv) & 1u) != 0;
        return any_mv ? WSTR_ERR_TOO_MANY_STATES : WSTR_ERR_UNSUPPORTED;
    }
    L.KC = kSplits[best_split].kc;
    L.KG = kSplits[best_split].kg;
    const int K = L.KC + L.KG, NP = 32 * K;
    L.state_of_pos.assign(NP, -1);
    L.pos_of_state.assign(S, -1);
    int lane = 0;
    std::vector<int> generic;
    for (size_t i = 0; i < c.seqs.size(); ++i) {
        const std::vector<int> &q = c.seqs[i];
        const int in_lanes = best_lanes[i] * L.KC;
        const int head = (int)q.size() - in_lanes;
        for (int n = 0; n < head; ++n) generic.push_back(q[n]);
        for (int n = head; n < (int)q.size(); ++n) {
            const int off = n - head;
            const int pos = (lane + off / L.KC) * K + off % L.KC;
            L.state_of_pos[pos] = q[n];
            L.pos_of_state[q[n]] = pos;
        }
        lane += best_lanes[i];
    }
    L.n_lanes = lane;
    std::sort(generic.begin(), generic.end());
    // "low" layout (dtw.cu: DegOf): when the generic states with more than one incoming edge fit
    // the last generic slot, all other generic slots are built with a single candidate
    std::vector<int> multi, single;
    for (int g : generic) (c.indeg[g] > 1 ? multi : single).push_back(g);
    const bool low = L.KG >= 2 && mv == 4 && (int)multi.size() <= 32 &&
                     (int)single.size() <= 32 * (L.KG - 1) + (32 - (int)multi.size());
    // "graded" layout: four candidates for the last slot, two for the one before it, one for the others --
    // when the states with three or four incoming edges fit the last slot and those with two the rest of it
    // plus the slot before
    std::vector<int> deg34, deg2;
    for (int g : multi) (c.indeg[g] > 2 ? deg34 : deg2).push_back(g);
    const int spare_last = 32 - (int)deg34.size();
    const int deg2_in_prev = std::max(0, (int)deg2.size() - std::max(spare_last, 0));
    const bool graded = !low && L.KG >= 3 && mv == 4 && (int)deg34.size() <= 32 && deg2_in_prev <= 32 &&
                        (int)single.size() <= 32 * (L.KG - 2) + (32 - deg2_in_prev) +
                                                  std::max(0, spare_last - (int)deg2.size());
    if (low) {
        // singles fill slots 0..KG-2 and then the free lanes of the last slot, in state order
        generic.clear();
        const int head = std::min<int>((int)single.size(), 32 * (L.KG - 1));
        generic.insert(generic.end(), single.begin(), single.begin() + head);
        generic.resize(32 * (L.KG - 1), -1);
        generic.insert(generic.end(), multi.begin(), multi.end());
        generic.insert(generic.end(), single.begin() + head, single.end());
    } else if (graded) {
        // last slot: the states with 3-4 incoming edges, then those with two; slot before: the rest of those
        // with two; singles fill slots 0..KG-3 and then whatever is free in the two others
        std::vector<int> last(deg34), prev;
        size_t d2 = 0;
        while (d2 < deg2.size() && (int)last.size() < 32) last.push_back(deg2[d2++]);
        while (d2 < deg2.size()) prev.push_back(deg2[d2++]);
        size_t s1 = std::min<size_t>(single.size(), 32 * (size_t)(L.KG - 2));
        generic.assign(single.begin(), single.begin() + s1);
        generic.resize(32 * (size_t)(L.KG - 2), -1);
        while (s1 < single.size() && (int)prev.size() < 32) prev.push_back(single[s1++]);
        while (s1 < single.size() && (int)last.size() < 32) last.push_back(single[s1++]);
        prev.resize(32, -1);
        generic.insert(generic.end(), prev.begin(), prev.end());
        generic.insert(generic.end(), last.begin(), last.end());
    }
    int max_indeg = 0;
    int placed = 0;
    for (size_t gi = 0; gi < generic.size(); ++gi) {
        if (generic[gi] < 0) continue;
        const int g = (int)gi / 32, ln = (int)gi % 32;
        const int pos = ln * K + L.KC + g;
        L.state_of_pos[pos] = generic[gi];
        L.pos_of_state[generic[gi]] = pos;
        max_indeg = std::max(max_indeg, c.indeg[generic[gi]]);
        ++placed;
    }
    L.n_generic = placed;
    if (max_indeg > WSTR_MAX_DEG) return WSTR_ERR_UNSUPPORTED;
    L.DEG = graded ? 242 : (max_indeg <= 2 ? 2 : 4) + (low ? 100 : 0);
    return WSTR_OK;
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

extern "C" int wstr_automaton_create(const double *values, const int32_t *seq_idx, const int32_t *in_ptr,
                                     const int32_t *in_idx, const uint8_t *rep_mask, const uint8_t *last_base,
                                     int32_t S, int32_t endstate, int32_t flank_length, int32_t mv,
                                     wstr_automaton **out) {
    if (!values || !seq_idx || !in_ptr || !out || S <= 0) return WSTR_ERR_INVALID_ARGUMENT;
    if (mv < 2) return WSTR_ERR_INVALID_ARGUMENT;           // reference: assert min_values_per_state > 1, config.py:115
    if (S <= mv) return WSTR_ERR_INVALID_ARGUMENT;          // reference: IndexError at caller.py:208
    if (endstate < 0 || endstate >= S) return WSTR_ERR_INVALID_ARGUMENT;
    if (S > 32767) return WSTR_ERR_TOO_MANY_STATES;         // traceback tables hold state indices in 15 bits
    const int E = in_ptr[S];
    if (E > 0 && !in_idx) return WSTR_ERR_INVALID_ARGUMENT;
    for (int e = 0; e < E; ++e)
        if (in_idx[e] < 0 || in_idx[e] >= S) return WSTR_ERR_INVALID_ARGUMENT;

    // the specialised register layout if there is one for this automaton and setting, else the
    // catch-all kernel (dtw_any.cu): nothing the reference accepts is refused
    Layout L;
    const bool any = g_generic_only || mv > WSTR_MAX_MV || build_layout(S, in_ptr, in_idx, mv, L) != WSTR_OK;
    const int spad = (S + 31) / 32 * 32;
    if (any) {
        for (int j = 0; j < S; ++j)
            if (in_ptr[j + 1] - in_ptr[j] > 254) return WSTR_ERR_UNSUPPORTED;      // one byte per direction code
        if (wstr_any_smem_bytes(mv, spad) > WSTR_ANY_SMEM_MAX) return WSTR_ERR_TOO_MANY_STATES;
        L.KC = L.KG = 0;
        L.DEG = 0;
        L.n_lanes = L.n_generic = 0;
        L.state_of_pos.clear();
        L.pos_of_state.assign(S, 0);
    }
    const int KC = L.KC, KG = L.KG, K = KC + KG, NP = 32 * K;
    const int inf_cell = KG * 32 + 32;

    // published-row index of every state (-1 = not readable by other lanes)
    auto published = [&](int state) {
        const int pos = L.pos_of_state[state];
        const int lane = pos / K, u = pos % K;
        if (u >= KC) return (u - KC) * 32 + lane;
        if (u == KC - 1) return KG * 32 + lane;
        return -1;
    };

    std::vector<uint32_t> lane_tab(32 * WSTR_LANE_TAB_STRIDE, 0u);
    std::vector<int32_t> pred_tab((size_t)NP * WSTR_PRED_STRIDE, -1);   // (state << 16) | position
    std::vector<double> v_pos(NP, 0.0);
    std::vector<int16_t> sop(NP, -1);
    const int boundary = flank_length - 10;
    const int after = seq_idx[S - 1] - boundary;     // caller.py:211-212
    for (int lane = 0; lane < 32; ++lane) {
        lane_tab[lane * WSTR_LANE_TAB_STRIDE + 1] = (uint32_t)inf_cell;
        for (int g = 0; g < WSTR_LANE_TAB_STRIDE - 2; ++g)
            lane_tab[lane * WSTR_LANE_TAB_STRIDE + 2 + g] = (uint32_t)inf_cell * 0x01010101u;
    }
    for (int pos = 0; pos < NP; ++pos) {
        const int lane = pos / K, u = pos % K;
        const int j = L.state_of_pos[pos];
        sop[pos] = (int16_t)j;
        if (j < 0) continue;
        v_pos[pos] = values[j];
        if (seq_idx[j] < after) lane_tab[lane * WSTR_LANE_TAB_STRIDE + 0] |= 1u << u;
        const int deg = in_ptr[j + 1] - in_ptr[j];
        if (u < KC) {
            if (deg > 1) return WSTR_ERR_UNSUPPORTED;          // cannot happen: layout invariant
            if (deg == 1) {
                const int pstate = in_idx[in_ptr[j]];
                const int ppos = L.pos_of_state[pstate];
                pred_tab[(size_t)pos * WSTR_PRED_STRIDE + 1] = (pstate << 16) | ppos;
                if (u == 0) {
                    const int q = published(pstate);
                    if (q < 0) return WSTR_ERR_UNSUPPORTED;    // layout invariant
                    lane_tab[lane * WSTR_LANE_TAB_STRIDE + 1] = (uint32_t)q;
                } else if (ppos != pos - 1) {
                    return WSTR_ERR_UNSUPPORTED;               // layout invariant
                }
            } else if (u != 0) {
                return WSTR_ERR_UNSUPPORTED;                   // a source state can only open a lane
            }
        } else {
            uint32_t packed = 0;
            for (int r = 0; r < WSTR_MAX_DEG; ++r) {
                int q = inf_cell;
                if (r < deg) {
                    const int pstate = in_idx[in_ptr[j] + r];
                    q = published(pstate);
                    if (q < 0) return WSTR_ERR_UNSUPPORTED;    // layout invariant
                    pred_tab[(size_t)pos * WSTR_PRED_STRIDE + 1 + r] = (pstate << 16) | L.pos_of_state[pstate];
                }
                packed |= (uint32_t)q << (8 * r);
            }
            lane_tab[lane * WSTR_LANE_TAB_STRIDE + 2 + (u - KC)] = packed;
        }
    }

    DevAutomaton d;
    memset(&d, 0, sizeof(d));
    // one device blob
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    const size_t o_v = take(sizeof(double) * NP), o_sop = take(sizeof(int16_t) * NP),
                 o_lt = take(sizeof(uint32_t) * lane_tab.size()), o_pt = take(sizeof(int32_t) * pred_tab.size()),
                 o_val = take(sizeof(double) * S), o_sq = take(sizeof(int32_t) * S), o_rm = take(S), o_lb = take(S),
                 o_ip = take(sizeof(int32_t) * (S + 1)), o_ii = take(sizeof(int32_t) * (size_t)std::max(E, 1));
    std::vector<unsigned char> blob(off, 0);
    memcpy(blob.data() + o_v, v_pos.data(), sizeof(double) * NP);
    memcpy(blob.data() + o_sop, sop.data(), sizeof(int16_t) * NP);
    memcpy(blob.data() + o_lt, lane_tab.data(), sizeof(uint32_t) * lane_tab.size());
    memcpy(blob.data() + o_pt, pred_tab.data(), sizeof(int32_t) * pred_tab.size());
    memcpy(blob.data() + o_val, values, sizeof(double) * S);
    memcpy(blob.data() + o_sq, seq_idx, sizeof(int32_t) * S);
    if (rep_mask) memcpy(blob.data() + o_rm, rep_mask, S);
    if (last_base) memcpy(blob.data() + o_lb, last_base, S);
    memcpy(blob.data() + o_ip, in_ptr, sizeof(int32_t) * (S + 1));
    if (E > 0) memcpy(blob.data() + o_ii, in_idx, sizeof(int32_t) * (size_t)E);

    void *d_blob = nullptr;
    WSTR_CUDA(cudaMalloc(&d_blob, off));
    cudaError_t ce = cudaMemcpy(d_blob, blob.data(), off, cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) {
        cudaFree(d_blob);
        return wstr_set_cuda_error(ce, "cudaMemcpy(automaton)");
    }
    unsigned char *base = static_cast<unsigned char *>(d_blob);
    d.v_pos = reinterpret_cast<const double *>(base + o_v);
    d.state_of_pos = reinterpret_cast<const int16_t *>(base + o_sop);
    d.lane_tab = reinterpret_cast<const uint32_t *>(base + o_lt);
    d.pred_tab = reinterpret_cast<const int32_t *>(base + o_pt);
    d.K = K;
    d.KC = KC;
    d.KG = KG;
    d.DEG = L.DEG;
    if (any) {                       // catch-all: one byte per cell, four rows per word (dtw_any.cu)
        d.NB = 8;
        d.RPW = 4;
    } else {                         // direction bits per lane and row (dtw.cu: DirFmt)
        if (L.DEG >= 200) d.NB = KC + (KG - 2) + (L.DEG - 200) % 10 + (L.DEG - 200) / 10;
        else if (L.DEG >= 100) d.NB = KC + (KG - 1) + (L.DEG - 100);
        else d.NB = KC + KG * L.DEG;
        d.RPW = 32 / d.NB;
    }
    d.S = S;
    d.end_pos = L.pos_of_state[endstate];
    d.values = reinterpret_cast<const double *>(base + o_val);
    d.seq_idx = reinterpret_cast<const int32_t *>(base + o_sq);
    d.in_ptr = reinterpret_cast<const int32_t *>(base + o_ip);
    d.in_idx = reinterpret_cast<const int32_t *>(base + o_ii);
    d.any = any ? 1 : 0;
    d.endstate = endstate;
    d.after = after;
    d.spad = spad;
    d.mv = mv;
    d.th1 = 6 * boundary;
    d.band6 = 6 * boundary;
    // The end band skips the states with seq_idx < after.  If none of them has an incoming edge
    // from a state outside that set, the skipped cells stay +inf on their own once the values
    // computed before the band have left the pipeline (mv rows), and the kernel drops the
    // per-cell band test from there on.
    d.band_closed = 1;
    for (int j = 0; j < S; ++j) {
        if (seq_idx[j] >= after) continue;
        for (int e = in_ptr[j]; e < in_ptr[j + 1]; ++e)
            if (seq_idx[in_idx[e]] >= after) d.band_closed = 0;
    }
    for (int c = 0; c <= mv && c <= WSTR_MAX_MV; ++c) d.init_pos[c] = L.pos_of_state[c];

    wstr_automaton *a = new wstr_automaton();
    a->dev = d;
    a->d_blob = d_blob;
    a->n_edges = E;
    a->n_generic = L.n_generic;
    a->n_chain_lanes = L.n_lanes;
    a->flank_length = flank_length;
    a->h_state_of_pos = new int32_t[NP];
    for (int p = 0; p < NP; ++p) a->h_state_of_pos[p] = L.state_of_pos[p];
    a->d_values = reinterpret_cast<const double *>(base + o_val);
    a->d_seq_idx = reinterpret_cast<const int32_t *>(base + o_sq);
    a->d_rep_mask = base + o_rm;
    a->d_last_base = base + o_lb;
    *out = a;
    return WSTR_OK;
}

extern "C" int wstr_set_generic_only(int32_t on) {
    g_generic_only = on != 0;
    return WSTR_OK;
}

extern "C" int wstr_automaton_plan(const int32_t *in_ptr, const int32_t *in_idx, int32_t S, int32_t mv,
                                   int32_t *info, int32_t *state_of_pos, int32_t n_pos) {
    if (!in_ptr || !info || S <= 0 || mv < 2) return WSTR_ERR_INVALID_ARGUMENT;
    Layout L;
    if (g_generic_only || mv > WSTR_MAX_MV || build_layout(S, in_ptr, in_idx, mv, L) != WSTR_OK) {
        // no specialised layout: the catch-all kernel takes it (dtw_any.cu)
        for (int j = 0; j < S; ++j)
            if (in_ptr[j + 1] - in_ptr[j] > 254) return WSTR_ERR_UNSUPPORTED;
        if (wstr_any_smem_bytes(mv, (S + 31) / 32 * 32) > WSTR_ANY_SMEM_MAX) return WSTR_ERR_TOO_MANY_STATES;
        for (int i = 0; i < 5; ++i) info[i] = 0;
        return WSTR_OK;
    }
    info[0] = L.KC;
    info[1] = L.KG;
    info[2] = L.DEG;
    info[3] = L.n_lanes;
    info[4] = L.n_generic;
    if (state_of_pos)
        for (int p = 0; p < n_pos && p < 32 * (L.KC + L.KG); ++p) state_of_pos[p] = L.state_of_pos[p];
    return WSTR_OK;
}

extern "C" int wstr_automaton_destroy(wstr_automaton *a) {
    if (!a) return WSTR_OK;
    cudaFree(a->d_blob);
    delete[] a->h_state_of_pos;
    delete a;
    return WSTR_OK;
}

extern "C" int wstr_automaton_info(const wstr_automaton *a, int32_t *info, int32_t n_info) {
    if (!a || !info) return WSTR_ERR_INVALID_ARGUMENT;
    const int32_t vals[9] = {a->dev.K,  a->dev.NB,  a->dev.KC,    a->dev.KG,          a->dev.S,
                             a->n_edges, a->n_generic, a->dev.band_closed, a->dev.DEG};
    for (int i = 0; i < n_info && i < 9; ++i) info[i] = vals[i];
    return WSTR_OK;
}

extern "C" int wstr_automaton_layout(const wstr_automaton *a, int32_t *state_of_pos, int32_t n_pos) {
    if (!a || !state_of_pos) return WSTR_ERR_INVALID_ARGUMENT;
    for (int p = 0; p < n_pos && p < 32 * a->dev.K; ++p) state_of_pos[p] = a->h_state_of_pos[p];
    return WSTR_OK;
}

// ------------------------------------------------------------------------------------------
// Host plan of a batch.  Everything the kernels need to know about the reads (automaton
// tables, per-read records, the longest-first processing order, the waves that fit the
// direction-code workspace) is laid out once per call in a pinned, device-mapped staging slot
// and brought into the workspace by a small copy kernel on the caller's stream -- not by the
// DMA engines, which a pipelining caller keeps busy with the next chunk's signal.  Nothing
// else crosses PCIe during the call and the host never waits for the device.
// ------------------------------------------------------------------------------------------
namespace {

struct StageSlot {
    void *h = nullptr;
    size_t cap = 0;
    cudaEvent_t done = nullptr;
    bool pending = false;     // its upload kernel may still be reading it
    bool reserved = false;    // handed out by stage_acquire, not yet committed
    int dev = -1;             // device its event belongs to (the pinned buffer itself is portable)
};
constexpr int kStageSlots = 8;
StageSlot g_stage[kStageSlots];
int g_stage_next = 0;
std::mutex g_stage_mu;
std::vector<void *> g_stage_parked;
size_t g_stage_parked_bytes = 0;

// a staging slot of at least `bytes`, free to overwrite.  A slot whose upload has completed is reused
// before a fresh one is allocated: pinning host memory costs milliseconds (and serialises in the
// kernel when several processes do it at once), so in steady state one or two slots do all the work.
int stage_acquire(size_t bytes, StageSlot **out) {
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_stage_mu);
    int pick = -1;
    for (int pass = 0; pass < 2 && pick < 0; ++pass) {
        for (int i = 0; i < kStageSlots && pick < 0; ++i) {
            StageSlot &sl = g_stage[i];
            if (sl.pending && cudaEventQuery(sl.done) == cudaSuccess) sl.pending = false;
            if (sl.pending || sl.reserved) continue;
            if (pass == 0 ? sl.cap >= bytes : true) pick = i;   // first a free slot that is large enough, then any free one
        }
    }
    if (pick < 0 && getenv("WSTR_DEBUG_TIMING")) {
        for (int i = 0; i < kStageSlots; ++i)
            fprintf(stderr, "[wstr stage] slot %d cap %zu pending %d reserved %d query %d\n", i, g_stage[i].cap,
                    (int)g_stage[i].pending, (int)g_stage[i].reserved,
                    g_stage[i].done ? (int)cudaEventQuery(g_stage[i].done) : -1);
    }
    if (pick < 0) {          // everything in flight: wait for the oldest
        for (int tries = 0; tries < kStageSlots && pick < 0; ++tries) {
            const int i = g_stage_next;
            g_stage_next = (g_stage_next + 1) % kStageSlots;
            if (!g_stage[i].reserved) pick = i;
        }
        if (pick < 0) return WSTR_ERR_INVALID_ARGUMENT;   // more concurrent calls than staging slots
        WSTR_CUDA(cudaEventSynchronize(g_stage[pick].done));
        g_stage[pick].pending = false;
    }
    StageSlot &sl = g_stage[pick];
    if (sl.cap < bytes) {
        // cudaFreeHost waits for the whole device: an outgrown buffer is parked and only freed once the
        // parked ones add up to more than the live one would need anyway (sizes double, so that is rare)
        if (sl.h) {
            g_stage_parked.push_back(sl.h);
            g_stage_parked_bytes += sl.cap;
        }
        sl.h = nullptr;
        sl.cap = 0;
        size_t cap = 1 << 16;
        while (cap < bytes) cap <<= 1;
        if (g_stage_parked_bytes > 4 * cap) {
            for (void *p : g_stage_parked) cudaFreeHost(p);
            g_stage_parked.clear();
            g_stage_parked_bytes = 0;
        }
        WSTR_CUDA(cudaHostAlloc(&sl.h, cap, cudaHostAllocMapped | cudaHostAllocPortable));
        sl.cap = cap;
    }
    if (sl.done && sl.dev != dev) {       // a slot last used from another device: its event cannot be recorded here
        cudaEventDestroy(sl.done);
        sl.done = nullptr;
    }
    if (!sl.done) WSTR_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    sl.dev = dev;
    sl.reserved = true;
    *out = &sl;
    return WSTR_OK;
}

void stage_release(StageSlot *sl) {   // a reserved slot that will not be committed after all
    std::lock_guard<std::mutex> lock(g_stage_mu);
    sl->reserved = false;
}

// work counters are cleared by a kernel, not cudaMemsetAsync: the driver may run a memset on a
// copy engine, behind whatever bulk copies a pipelining caller has queued there
__global__ void zero_kernel(int32_t *p, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = 0;
}
int zero_counters(int32_t *d, int n, cudaStream_t s) {
    zero_kernel<<<1, 64, 0, s>>>(d, n);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}

__global__ void upload_kernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, size_t n16) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// staged bytes -> device, on the stream; the slot is reusable once `done` has passed
int stage_upload(StageSlot *sl, void *d_dst, size_t bytes, cudaStream_t s) {
    const size_t n16 = (bytes + 15) / 16;
    const int grid = (int)std::min<size_t>((n16 + 255) / 256, 512);
    void *d_src = nullptr;
    WSTR_CUDA(cudaHostGetDevicePointer(&d_src, sl->h, 0));
    wstr_prof_begin(4, s);
    upload_kernel<<<grid, 256, 0, s>>>(static_cast<uint4 *>(d_dst), static_cast<const uint4 *>(d_src), n16);
    wstr_prof_end(s);
    WSTR_CUDA(cudaGetLastError());
    const cudaError_t ee = cudaEventRecord(sl->done, s);
    {
        std::lock_guard<std::mutex> lock(g_stage_mu);
        sl->pending = ee == cudaSuccess;
        sl->reserved = false;
    }
    if (ee != cudaSuccess) return wstr_set_cuda_error(ee, "cudaEventRecord(stage)");
    return WSTR_OK;
}

}  // namespace

// the same staging for the other entry points of the library (aux.cu)
int wstr_stage_begin(size_t bytes, void **h_ptr, void **token) {
    StageSlot *sl = nullptr;
    const int rc = stage_acquire(bytes, &sl);
    if (rc != WSTR_OK) return rc;
    *h_ptr = sl->h;
    *token = sl;
    return WSTR_OK;
}
int wstr_stage_commit(void *token, void *d_dst, size_t bytes, cudaStream_t s) {
    return stage_upload(static_cast<StageSlot *>(token), d_dst, bytes, s);
}
namespace {
__global__ void zero16_kernel(uint4 *__restrict__ p, size_t n16) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        p[i] = make_uint4(0u, 0u, 0u, 0u);
}
}  // namespace
// d 16-byte aligned, bytes a multiple of 16
int wstr_zero_async(void *d, size_t bytes, cudaStream_t s) {
    const size_t n16 = bytes / 16;
    if (n16 == 0) return WSTR_OK;
    const int grid = (int)std::min<size_t>((n16 + 255) / 256, 148 * 8);
    zero16_kernel<<<grid, 256, 0, s>>>(static_cast<uint4 *>(d), n16);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}

namespace {

inline int64_t dir_words(const wstr_automaton *a, int T) {   // RPW rows share a word per lane (dtw.cu: DirFmt)
    if (a->dev.any) return ((int64_t)T + 3) / 4 * a->dev.spad;   // ... per state in the catch-all (dtw_any.cu)
    return ((int64_t)T + a->dev.RPW - 1) / a->dev.RPW * 32;
}

struct FillLaunch {
    int kc, kg, deg;   // 0, 0, 0: the catch-all kernel
    int spad_max;      // catch-all: widest automaton of the launch
    int begin, n;      // slice of the order array
    int counter;       // index of its work counter
};
struct Wave {
    std::vector<FillLaunch> launches;
};

// block uploaded per call: [DevAutomaton x A][ReadMeta x n][order x n] (+ the mid-stage tables)
struct BlockLayout {
    size_t o_auts, o_meta, o_order, o_mauts, o_reads, bytes;
};
BlockLayout block_layout(int n_automata, int n_reads, bool with_mid) {
    BlockLayout b;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    b.o_auts = take(sizeof(DevAutomaton) * (size_t)n_automata);
    b.o_meta = take(sizeof(ReadMeta) * (size_t)n_reads);
    b.o_order = take(sizeof(int32_t) * (size_t)n_reads);
    b.o_mauts = take(with_mid ? sizeof(MidAutomaton) * (size_t)n_automata : 0);
    b.o_reads = take(with_mid ? sizeof(MidRead) * (size_t)n_reads : 0);
    b.bytes = off;
    return b;
}

constexpr int kCounters = 64;   // work counters per wave (one per kernel shape present)

// Fill the DP part of the block and cut the batch into waves.  mask_off may be NULL.
int plan_fill(wstr_automaton *const *automata, int n_automata, const int32_t *read_automaton, const int64_t *sig_off,
              const int32_t *lengths, const int64_t *mask_off, int n_reads, int64_t dir_capacity,
              unsigned char *block, const BlockLayout &bl, std::vector<Wave> &waves) {
    DevAutomaton *h_auts = reinterpret_cast<DevAutomaton *>(block + bl.o_auts);
    ReadMeta *meta = reinterpret_cast<ReadMeta *>(block + bl.o_meta);
    int32_t *order = reinterpret_cast<int32_t *>(block + bl.o_order);
    for (int a = 0; a < n_automata; ++a) h_auts[a] = automata[a]->dev;

    // longest reads first, equal lengths in batch order: a counting sort over the lengths (a comparison
    // sort of a million reads is tens of milliseconds of host time in front of every call)
    std::vector<int> idx(n_reads);
    int maxlen = 0;
    for (int r = 0; r < n_reads; ++r) maxlen = std::max(maxlen, (int)lengths[r]);
    if (maxlen <= (1 << 22)) {
        std::vector<int> pos((size_t)maxlen + 2, 0);
        for (int r = 0; r < n_reads; ++r) pos[lengths[r]]++;
        int run = 0;
        for (int l = maxlen; l >= 0; --l) {       // first slot of each length, longest first
            const int c = pos[l];
            pos[l] = run;
            run += c;
        }
        for (int r = 0; r < n_reads; ++r) idx[pos[lengths[r]]++] = r;
    } else {
        std::iota(idx.begin(), idx.end(), 0);
        std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return lengths[x] > lengths[y]; });
    }

    // kernel shape class of every automaton
    std::vector<int> cls_of(n_automata), cls_rep, cls_spad;
    for (int a = 0; a < n_automata; ++a) {
        const DevAutomaton &d = automata[a]->dev;
        int c = -1;
        for (size_t k = 0; k < cls_rep.size(); ++k) {
            const DevAutomaton &o = automata[cls_rep[k]]->dev;
            if (o.KC == d.KC && o.KG == d.KG && o.DEG == d.DEG) c = (int)k;
        }
        if (c < 0) {
            c = (int)cls_rep.size();
            cls_rep.push_back(a);
            cls_spad.push_back(0);
        }
        cls_spad[c] = std::max(cls_spad[c], (int)d.spad);
        cls_of[a] = c;
    }
    const int n_classes = (int)cls_rep.size();
    std::vector<int> cls_first, cls_count, cls_order;

    waves.clear();
    int cursor = 0;
    while (cursor < n_reads) {
        const int wave_begin = cursor;
        int64_t used = 0;
        while (cursor < n_reads) {
            const int r = idx[cursor];
            const int a = read_automaton ? read_automaton[r] : 0;
            const int64_t need = dir_words(automata[a], lengths[r]);
            if (used + need > dir_capacity) break;
            ReadMeta &m = meta[cursor];
            m.sig_off = sig_off[r];
            m.dir_off = used;
            m.mask_off = mask_off ? mask_off[r] : 0;
            m.T = lengths[r];
            m.aut = a;
            m.read = r;
            m.pad_ = 0;
            used += need;
            ++cursor;
        }
        if (cursor == wave_begin) return WSTR_ERR_WORKSPACE_TOO_SMALL;   // one read does not fit
        // one launch per kernel shape (chain slots, generic slots, in-degree) present in this wave, shapes in
        // order of first appearance, the reads of a shape in wave order (longest first): two passes over the
        // wave with the automata's shape classes looked up from a small table
        Wave w;
        const int nw = cursor - wave_begin;
        cls_first.assign(n_classes, -1);
        cls_count.assign(n_classes, 0);
        cls_order.clear();
        for (int i = 0; i < nw; ++i) {
            const int c = cls_of[meta[wave_begin + i].aut];
            if (cls_count[c]++ == 0) cls_order.push_back(c);
        }
        int filled = wave_begin;
        for (int c : cls_order) {
            const DevAutomaton &ref = automata[cls_rep[c]]->dev;
            FillLaunch fl;
            fl.kc = ref.KC;
            fl.kg = ref.KG;
            fl.deg = ref.DEG;
            fl.spad_max = cls_spad[c];
            fl.begin = filled;
            fl.n = cls_count[c];
            fl.counter = (int)w.launches.size();
            if (fl.counter >= kCounters) return WSTR_ERR_UNSUPPORTED;
            w.launches.push_back(fl);
            cls_first[c] = filled;
            filled += cls_count[c];
        }
        for (int i = 0; i < nw; ++i) order[cls_first[cls_of[meta[wave_begin + i].aut]]++] = wave_begin + i;
        waves.push_back(std::move(w));
    }
    return WSTR_OK;
}

struct FillDevice {
    const DevAutomaton *auts;
    const ReadMeta *meta;
    const int32_t *order;
    int32_t *counters;    // kCounters ints
    uint32_t *dir;
};

// one DP pass (fill + traceback) over the planned waves; no host<->device traffic
int run_fill(const std::vector<Wave> &waves, const FillDevice &fd, int mv, const double *d_signal,
             const uint32_t *d_maskbits, int32_t *d_trace, double *d_end_cost, int32_t *d_status, int respect_status,
             cudaStream_t s) {
    for (const Wave &w : waves) {
        if (int zrc = zero_counters(fd.counters, kCounters, s)) return zrc;
        for (const FillLaunch &fl : w.launches) {
            FillParams fp;
            fp.auts = fd.auts;
            fp.meta = fd.meta;
            fp.order = fd.order + fl.begin;
            fp.n = fl.n;
            fp.queue = fd.counters + fl.counter;
            fp.signal = d_signal;
            fp.maskbits = d_maskbits;
            fp.dir = fd.dir;
            fp.trace = d_trace;
            fp.end_cost = d_end_cost;
            fp.status = d_status;
            fp.respect_status = respect_status;
            wstr_prof_begin(0, s);
            const int rc = fl.kc + fl.kg == 0 ? wstr_launch_fill_any(mv, fl.spad_max, fp, s)
                                              : wstr_launch_fill(fl.kc, fl.kg, fl.deg, mv, fp, s);
            wstr_prof_end(s);
            if (rc != WSTR_OK) return rc;
        }
    }
    return WSTR_OK;
}

int check_reads(wstr_automaton *const *automata, int n_automata, const int32_t *read_automaton, const int64_t *sig_off,
                const int32_t *lengths, int n_reads) {
    const int mv = automata[0]->dev.mv;
    for (int a = 0; a < n_automata; ++a)
        if (!automata[a] || automata[a]->dev.mv != mv) return WSTR_ERR_INVALID_ARGUMENT;
    for (int r = 0; r < n_reads; ++r) {
        const int a = read_automaton ? read_automaton[r] : 0;
        if (a < 0 || a >= n_automata || lengths[r] < 0 || (sig_off[r] & 1)) return WSTR_ERR_INVALID_ARGUMENT;
    }
    return WSTR_OK;
}

// workspace of a stand-alone pass: [counters][block][direction codes]
struct WarpWs {
    size_t o_counters, o_block, o_dir;
    BlockLayout bl;
};
WarpWs plan_warp_ws(int n_automata, int n_reads) {
    WarpWs w;
    w.bl = block_layout(n_automata, n_reads, false);
    w.o_counters = 0;
    w.o_block = 256;
    w.o_dir = align_up(w.o_block + w.bl.bytes, 256);
    return w;
}

}  // namespace

extern "C" int64_t wstr_warp_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                             const int32_t *read_automaton, const int32_t *lengths,
                                             int32_t n_reads) {
    if (!automata || n_automata <= 0 || n_reads < 0) return WSTR_ERR_INVALID_ARGUMENT;
    const WarpWs w = plan_warp_ws(n_automata, n_reads);
    int64_t words = 0;
    for (int r = 0; r < n_reads; ++r) {
        const int a = read_automaton ? read_automaton[r] : 0;
        if (a < 0 || a >= n_automata) return WSTR_ERR_INVALID_ARGUMENT;
        words += dir_words(automata[a], lengths[r]);
    }
    return (int64_t)w.o_dir + words * 4 + 256;
}

extern "C" int wstr_warp_batch(wstr_automaton *const *automata, int32_t n_automata,
                               const int32_t *read_automaton, const double *d_signal, const int64_t *sig_off,
                               const int32_t *lengths, const uint32_t *d_maskbits, const int64_t *mask_off,
                               int32_t n_reads, void *d_workspace, int64_t workspace_bytes, int32_t *d_trace,
                               double *d_end_cost, int32_t *d_status, void *stream) {
    if (!automata || n_automata <= 0 || n_reads < 0 || !d_signal || !sig_off || !lengths || !d_workspace ||
        !d_trace || !d_status)
        return WSTR_ERR_INVALID_ARGUMENT;
    if (d_maskbits && !mask_off) return WSTR_ERR_INVALID_ARGUMENT;
    if (n_reads == 0) return WSTR_OK;
    int rc = check_reads(automata, n_automata, read_automaton, sig_off, lengths, n_reads);
    if (rc != WSTR_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const WarpWs w = plan_warp_ws(n_automata, n_reads);
    if ((int64_t)w.o_dir >= workspace_bytes) return WSTR_ERR_WORKSPACE_TOO_SMALL;
    unsigned char *ws = static_cast<unsigned char *>(d_workspace);

    StageSlot *slot = nullptr;
    rc = stage_acquire(w.bl.bytes, &slot);
    if (rc != WSTR_OK) return rc;
    std::vector<Wave> waves;
    rc = plan_fill(automata, n_automata, read_automaton, sig_off, lengths, d_maskbits ? mask_off : nullptr, n_reads,
                   (workspace_bytes - (int64_t)w.o_dir) / 4, static_cast<unsigned char *>(slot->h), w.bl, waves);
    if (rc != WSTR_OK) {
        stage_release(slot);
        return rc;
    }
    rc = stage_upload(slot, ws + w.o_block, w.bl.bytes, s);
    if (rc != WSTR_OK) return rc;

    FillDevice fd;
    fd.auts = reinterpret_cast<const DevAutomaton *>(ws + w.o_block + w.bl.o_auts);
    fd.meta = reinterpret_cast<const ReadMeta *>(ws + w.o_block + w.bl.o_meta);
    fd.order = reinterpret_cast<const int32_t *>(ws + w.o_block + w.bl.o_order);
    fd.counters = reinterpret_cast<int32_t *>(ws + w.o_counters);
    fd.dir = reinterpret_cast<uint32_t *>(ws + w.o_dir);
    return run_fill(waves, fd, automata[0]->dev.mv, d_signal, d_maskbits, d_trace, d_end_cost, d_status, 0, s);
}

// ------------------------------------------------------------------------------------------
// whole per-read call: pass 1 -> mid-stage -> pass 2 -> mid-stage
// ------------------------------------------------------------------------------------------
namespace {

struct CallPlan {
    size_t o_counters, o_queue, o_block, o_state, o_cubic, o_resc, o_trace, o_mask, o_scratch, o_dir;
    BlockLayout bl;
    int64_t extent;       // elements of the signal buffer in use
    int64_t mask_words;
    int64_t scratch_bytes;
};

CallPlan plan_call(int n_automata, int n_reads, const int64_t *sig_off, const int32_t *lengths, int mv,
                   bool own_resc, bool own_trace, int reps = 0, int s_max = 0) {
    CallPlan c;
    c.extent = 0;
    c.mask_words = 0;
    c.scratch_bytes = 0;
    int64_t run_off = 0;
    for (int r = 0; r < n_reads; ++r) {
        const int64_t so = sig_off ? sig_off[r] : run_off;
        c.extent = std::max<int64_t>(c.extent, so + lengths[r] + 2);
        run_off += ((int64_t)lengths[r] + 1) & ~(int64_t)1;
        c.mask_words += (lengths[r] + 31) / 32;
        c.scratch_bytes += wstr_mid_scratch_bytes(lengths[r], mv, reps, s_max);
    }
    c.bl = block_layout(n_automata, n_reads, true);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    c.o_counters = take(kCounters * sizeof(int32_t));
    c.o_queue = take(256);
    c.o_block = take(c.bl.bytes);
    c.o_state = take(sizeof(MidState) * (size_t)n_reads);
    c.o_cubic = take(sizeof(double) * 8 * (size_t)n_reads);
    c.o_resc = take(own_resc ? sizeof(double) * (size_t)c.extent : 0);
    c.o_trace = take(own_trace ? sizeof(int32_t) * (size_t)c.extent : 0);
    c.o_mask = take(sizeof(uint32_t) * (size_t)(c.mask_words + 1));
    c.o_scratch = take((size_t)c.scratch_bytes);
    c.o_dir = off;
    return c;
}

}  // namespace

extern "C" int64_t wstr_call_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                             const int32_t *read_automaton, const int32_t *lengths,
                                             int32_t n_reads) {
    if (!automata || n_automata <= 0 || n_reads < 0 || !lengths) return WSTR_ERR_INVALID_ARGUMENT;
    int64_t words = 0;
    for (int r = 0; r < n_reads; ++r) {
        const int a = read_automaton ? read_automaton[r] : 0;
        if (a < 0 || a >= n_automata) return WSTR_ERR_INVALID_ARGUMENT;
        words += dir_words(automata[a], lengths[r]);
    }
    // (sized for rescaling.reps_as_one as well, which needs 8 more bytes per sample of scratch: the
    // parameters of the call are not known here)
    int s_max = 0;
    for (int a = 0; a < n_automata; ++a) s_max = std::max(s_max, (int)automata[a]->dev.S);
    const CallPlan c = plan_call(n_automata, n_reads, nullptr, lengths, automata[0]->dev.mv, true, true, 1, s_max);
    return (int64_t)c.o_dir + words * 4 + 256;
}

extern "C" int64_t wstr_call_workspace_min_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                                 const int32_t *read_automaton, const int32_t *lengths,
                                                 int32_t n_reads) {
    if (!automata || n_automata <= 0 || n_reads < 0 || !lengths) return WSTR_ERR_INVALID_ARGUMENT;
    int64_t widest = 0;
    for (int r = 0; r < n_reads; ++r) {
        const int a = read_automaton ? read_automaton[r] : 0;
        if (a < 0 || a >= n_automata) return WSTR_ERR_INVALID_ARGUMENT;
        widest = std::max(widest, dir_words(automata[a], lengths[r]));
    }
    int s_max = 0;
    for (int a = 0; a < n_automata; ++a) s_max = std::max(s_max, (int)automata[a]->dev.S);
    const CallPlan c = plan_call(n_automata, n_reads, nullptr, lengths, automata[0]->dev.mv, true, true, 1, s_max);
    return (int64_t)c.o_dir + widest * 4 + 256;
}

namespace {
struct HostTimer {      // WSTR_DEBUG_TIMING=1: host milliseconds of the sections of a call, on stderr
    bool on;
    std::chrono::steady_clock::time_point t0;
    const char *what;
    HostTimer(const char *w) : on(getenv("WSTR_DEBUG_TIMING") != nullptr), t0(std::chrono::steady_clock::now()), what(w) {}
    void lap(const char *label) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[wstr %s] %s %.3f ms\n", what, label, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};
}  // namespace

extern "C" int wstr_call_batch(wstr_automaton *const *automata, int32_t n_automata,
                               const int32_t *read_automaton, const uint8_t *read_reverse,
                               const double *d_signal, const int64_t *sig_off, const int32_t *lengths,
                               int32_t n_reads, const wstr_call_params *params, void *d_workspace,
                               int64_t workspace_bytes, const wstr_call_outputs *out, void *stream) {
    if (!automata || n_automata <= 0 || n_reads < 0 || !d_signal || !sig_off || !lengths || !params || !out ||
        !d_workspace || !out->d_len1 || !out->d_len2 || !out->d_cost1 || !out->d_cost2 || !out->d_status)
        return WSTR_ERR_INVALID_ARGUMENT;
    if ((out->d_seq1 || out->d_seq2) && !out->seq_off) return WSTR_ERR_INVALID_ARGUMENT;
    if (n_reads == 0) return WSTR_OK;
    if (params->method != 0 && params->method != 1) return WSTR_ERR_UNSUPPORTED;
    const int reps = params->reps_as_one != 0;
    int s_max = 0;
    for (int a = 0; a < n_automata; ++a)
        if (automata[a]) s_max = std::max(s_max, (int)automata[a]->dev.S);
    if (params->states_in_segment < 2) return WSTR_ERR_INVALID_ARGUMENT;
    const int mv = automata[0]->dev.mv;
    if (params->min_values_per_state != mv) return WSTR_ERR_INVALID_ARGUMENT;
    int rc = check_reads(automata, n_automata, read_automaton, sig_off, lengths, n_reads);
    if (rc != WSTR_OK) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool own_resc = out->d_rescaled == nullptr;
    const bool own_trace = out->d_trace1 == nullptr || out->d_trace2 == nullptr;
    const CallPlan c = plan_call(n_automata, n_reads, sig_off, lengths, mv, own_resc, own_trace, reps, s_max);
    if ((int64_t)c.o_dir >= workspace_bytes) return WSTR_ERR_WORKSPACE_TOO_SMALL;
    unsigned char *ws = static_cast<unsigned char *>(d_workspace);
    unsigned char *d_block = ws + c.o_block;
    int32_t *d_queue = reinterpret_cast<int32_t *>(ws + c.o_queue);
    MidState *d_state = reinterpret_cast<MidState *>(ws + c.o_state);
    double *d_cubic = reinterpret_cast<double *>(ws + c.o_cubic);
    double *d_resc = own_resc ? reinterpret_cast<double *>(ws + c.o_resc) : out->d_rescaled;
    int32_t *d_own_trace = reinterpret_cast<int32_t *>(ws + c.o_trace);
    int32_t *d_trace1 = out->d_trace1 ? out->d_trace1 : d_own_trace;
    int32_t *d_trace2 = out->d_trace2 ? out->d_trace2 : d_own_trace;
    uint32_t *d_mask = reinterpret_cast<uint32_t *>(ws + c.o_mask);
    unsigned char *d_scratch = ws + c.o_scratch;

    // ---- the whole host plan, staged and uploaded in one piece -----------------------------
    HostTimer timer("call_batch");
    StageSlot *slot = nullptr;
    rc = stage_acquire(c.bl.bytes, &slot);
    if (rc != WSTR_OK) return rc;
    timer.lap("stage_acquire");
    unsigned char *block = static_cast<unsigned char *>(slot->h);
    MidAutomaton *mauts = reinterpret_cast<MidAutomaton *>(block + c.bl.o_mauts);
    for (int a = 0; a < n_automata; ++a) {
        mauts[a].values = automata[a]->d_values;
        mauts[a].seq_idx = automata[a]->d_seq_idx;
        mauts[a].rep_mask = automata[a]->d_rep_mask;
        mauts[a].last_base = automata[a]->d_last_base;
        mauts[a].flank_length = automata[a]->flank_length;
        mauts[a].n_states = automata[a]->dev.S;
    }
    MidRead *reads = reinterpret_cast<MidRead *>(block + c.bl.o_reads);
    std::vector<int64_t> mask_off(n_reads);
    int64_t mo = 0, so = 0;
    for (int r = 0; r < n_reads; ++r) {
        MidRead &m = reads[r];
        m.sig_off = sig_off[r];
        m.mask_off = mo;
        m.ws_off = so;
        m.seq_off = out->seq_off ? out->seq_off[r] : -1;
        m.T = lengths[r];
        m.aut = read_automaton ? read_automaton[r] : 0;
        m.read = r;
        m.reverse = read_reverse ? (read_reverse[r] != 0) : 0;
        m.run_cap = lengths[r] / (mv > 2 ? mv - 1 : 1) + 16;
        m.pad_ = 0;
        mask_off[r] = mo;
        mo += (lengths[r] + 31) / 32;
        so += wstr_mid_scratch_bytes(lengths[r], mv, reps, s_max);
    }
    std::vector<Wave> waves;
    rc = plan_fill(automata, n_automata, read_automaton, sig_off, lengths, mask_off.data(), n_reads,
                   (workspace_bytes - (int64_t)c.o_dir) / 4, block, c.bl, waves);
    if (rc != WSTR_OK) {
        stage_release(slot);
        return rc;
    }
    timer.lap("plan");
    rc = stage_upload(slot, d_block, c.bl.bytes, s);
    if (rc != WSTR_OK) return rc;
    timer.lap("stage_upload");

    FillDevice fd;
    fd.auts = reinterpret_cast<const DevAutomaton *>(d_block + c.bl.o_auts);
    fd.meta = reinterpret_cast<const ReadMeta *>(d_block + c.bl.o_meta);
    fd.order = reinterpret_cast<const int32_t *>(d_block + c.bl.o_order);
    fd.counters = reinterpret_cast<int32_t *>(ws + c.o_counters);
    fd.dir = reinterpret_cast<uint32_t *>(ws + c.o_dir);

    // ---- first pass --------------------------------------------------------------------------
    rc = run_fill(waves, fd, mv, d_signal, nullptr, d_trace1, nullptr, out->d_status, 0, s);
    if (rc != WSTR_OK) return rc;
    MidParams mp;
    mp.auts = reinterpret_cast<const MidAutomaton *>(d_block + c.bl.o_mauts);
    mp.reads = reinterpret_cast<const MidRead *>(d_block + c.bl.o_reads);
    mp.n = n_reads;
    mp.queue = d_queue;
    mp.x = d_signal;
    mp.trace = d_trace1;
    mp.rescaled = d_resc;
    mp.maskbits = d_mask;
    mp.scratch = d_scratch;
    mp.state = d_state;
    mp.cubic = d_cubic;
    mp.len = out->d_len1;
    mp.cost = out->d_cost1;
    mp.seq = out->d_seq1;
    mp.status = out->d_status;
    mp.mv = mv;
    mp.sis = params->states_in_segment;
    mp.method = params->method;
    mp.reps = reps;
    mp.s_max = s_max;
    mp.pipe_ok = 1;
    for (int r = 0; r < n_reads; ++r)
        if (2 * (lengths[r] / (mv > 2 ? mv - 1 : 1) + 16) > lengths[r]) mp.pipe_ok = 0;
    mp.threshold = params->threshold;
    mp.max_std = params->max_std;
    mp.ties = out->d_ttest_ties;
    mp.tie_ulps = params->ttest_guard_ulps > 0 ? params->ttest_guard_ulps : 16;
    if (int zrc = zero_counters(d_queue, 64, s)) return zrc;
    wstr_prof_begin(1, s);
    rc = wstr_launch_midstage(mp, false, s);
    wstr_prof_end(s);
    if (rc != WSTR_OK) return rc;

    // ---- second pass on the rescaled signal, masked rows allow the shorter dwell ----------------
    rc = run_fill(waves, fd, mv, d_resc, d_mask, d_trace2, nullptr, out->d_status, 1, s);
    if (rc != WSTR_OK) return rc;
    mp.x = d_resc;
    mp.trace = d_trace2;
    mp.rescaled = nullptr;
    mp.maskbits = nullptr;
    mp.ties = nullptr;
    mp.len = out->d_len2;
    mp.cost = out->d_cost2;
    mp.seq = out->d_seq2;
    if (int zrc = zero_counters(d_queue, 64, s)) return zrc;
    wstr_prof_begin(1, s);
    rc = wstr_launch_midstage(mp, true, s);
    wstr_prof_end(s);
    timer.lap("launches");
    return rc;
}
