// (3c) Reads of a panel found in a whole run by their flanks (DESIGN.md section 4.6).
//
// Each locus of a panel has four chain automata: its template-strand left and right flank and its
// reverse-strand left and right flank.  Every one is searched in every whole normalised read with the window
// search of locate.cu (wso_locate's recurrence, operation order, tie rules and start-row tags), and a read
// belongs to a locus when both flanks of one strand are found, in order.
//
// locate_group_kernel: one CTA per (read, group).  A group is a run of whole loci (four automata each, in
// panel order) whose states, rings, published rows and edge lists fit GROUP_SMEM together; the threads own the
// states of the group's concatenated state list (thread t: t, t+NT, ...), each component keeping its own start
// state (its state 0) and end state.  The signal tile is fetched once per row for the whole group and there is
// one __syncthreads per row for the whole group, so many small automata share one pass over the read instead
// of one CTA, one pass and one barrier per row each.  A group whose rings alone do not fit keeps them in a
// slab of the workspace per CTA, as locate_kernel does.
//
// assign_reduce_kernel: one thread per (read, locus) applies the decision rule (assign.choose_loci is its
// host statement) to the four searches and appends a hit to a compact list, so the [read x chain] table never
// has to leave the device.
#include <algorithm>
#include <vector>

#include "wstr_internal.h"

namespace {

// 256 threads and 113 KB per group: two CTAs (16 warps) per SM.  A 12-chain group (three loci) is ~1 260
// states, ~5 per thread and row.  See DESIGN.md section 4.6 for the registers and the measurement.
constexpr int NT = 256;
constexpr int TILE = NT;                        // samples per signal tile: one per thread
constexpr size_t SMEM_MAX = 226 * 1024;         // sm_100's 227 KB opt-in, less the static part
constexpr size_t GROUP_SMEM = 113 * 1024;       // a group's budget, rings included
constexpr int CHAINS = 4;                       // automata per locus

struct GroupDesc {
    int32_t G, E, C, comp0;      // states, edges, components, first entry in the component table
    int32_t ring_gmem, pad_;     // rings in the CTA's workspace slab
};

struct GroupComp {
    int32_t aut, base, ebase, pad_;   // automaton; its first state and first edge in the group's lists
};

struct AsgItem {
    int64_t sig_off;
    int32_t T, read, group, pad_;
};

struct AsgParams {
    const DevAutomaton *auts;
    const GroupDesc *groups;
    const GroupComp *comps;
    const AsgItem *items;        // longest read first, a read's groups adjacent
    int32_t n;
    int32_t n_aut;
    int32_t *queue;              // zero when the plan arrives
    const double *signal;
    double offset;
    double *score;               // table [read * n_aut + automaton], struct of arrays
    int32_t *lo, *hi, *status;
    unsigned char *ring_gmem;    // slab of ring_slab bytes per CTA (groups with ring_gmem)
    int64_t ring_slab;
};

__host__ __device__ inline size_t ring_bytes(int mv, int G) { return (size_t)mv * G * (sizeof(double) + sizeof(int32_t)); }
// doubles: [ring mv x G (in shared memory)][pub 2 x G][v G][signal 2 x TILE][best C]
// int32:   [ring tags mv x G (in shared memory)][pub tags 2 x G][in_ptr G+1][in_idx E][flags G][lo C][hi C]
__host__ __device__ inline size_t group_smem(int mv, int G, int E, int C, bool rings) {
    const size_t r = rings ? (size_t)mv * G : 0;
    return sizeof(double) * (r + 3 * (size_t)G + 2 * TILE + C) +
           sizeof(int32_t) * (r + 2 * (size_t)G + (G + 1) + E + G + 2 * (size_t)C) + 16;
}

__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }

__global__ void __launch_bounds__(NT) locate_group_kernel(const AsgParams p, const int mv) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_next;
    const int tid = threadIdx.x;
    const double INF = dinf();
    const double lam = p.offset;

    for (;;) {
        __syncthreads();       // the previous item is done with shared memory
        if (tid == 0) s_next = atomicAdd(p.queue, 1);
        __syncthreads();
        const int it = s_next;
        if (it >= p.n) break;
        const AsgItem m = p.items[it];
        const GroupDesc gd = p.groups[m.group];
        const int G = gd.G, C = gd.C, T = m.T;
        double *dp = reinterpret_cast<double *>(smem_raw);
        double *ring;
        int32_t *rtag;
        if (gd.ring_gmem) {
            ring = reinterpret_cast<double *>(p.ring_gmem + (size_t)blockIdx.x * p.ring_slab);   // [mv][G]
            rtag = reinterpret_cast<int32_t *>(ring + (size_t)mv * G);
        } else {
            ring = dp;
            dp += (size_t)mv * G;
        }
        double *pub = dp;                 // [2][G]
        double *sv = pub + 2 * (size_t)G;
        double *sx = sv + G;              // [2][TILE]
        double *sbest = sx + 2 * TILE;    // [C]
        int32_t *ip = reinterpret_cast<int32_t *>(sbest + C);
        if (!gd.ring_gmem) {
            rtag = ip;
            ip += (size_t)mv * G;
        }
        int32_t *ptag = ip;               // [2][G]
        int32_t *sptr = ptag + 2 * (size_t)G;
        int32_t *sidx = sptr + G + 1;
        int32_t *sflag = sidx + gd.E;     // bit 0: a path may start here; >> 1: 1 + component it ends
        int32_t *slo = sflag + G;
        int32_t *shi = slo + C;

        // the group's concatenated state list, its edges in group indices, and no row yet
        for (int c = 0; c < C; ++c) {
            const GroupComp gc = p.comps[gd.comp0 + c];
            const DevAutomaton *A = p.auts + gc.aut;
            const int S = A->S, endstate = A->endstate;
            for (int j = tid; j < S; j += NT) {
                const int g = gc.base + j;
                sv[g] = __ldg(A->values + j);
                sptr[g] = gc.ebase + __ldg(A->in_ptr + j);
                sflag[g] = (j == 0 ? 1 : 0) | (j == endstate ? (c + 1) << 1 : 0);
            }
            const int nE = __ldg(A->in_ptr + S);
            for (int q = tid; q < nE; q += NT) sidx[gc.ebase + q] = gc.base + __ldg(A->in_idx + q);
        }
        if (tid == 0) sptr[G] = gd.E;
        for (int c = tid; c < C; c += NT) {
            sbest[c] = INF;
            slo[c] = -1;
            shi[c] = -1;
        }
        for (int g = tid; g < G; g += NT) {
            for (int s = 0; s < mv; ++s) ring[(size_t)s * G + g] = INF;
            pub[g] = INF;
            pub[G + g] = INF;
        }
        const double *gx = p.signal + m.sig_off;
        const int ntiles = (T + TILE - 1) / TILE;
        sx[tid] = tid < T ? gx[tid] : 0.0;
        __syncthreads();

        int slot = 0;            // i mod mv
        for (int c = 0; c < ntiles; ++c) {
            const int i_begin = c * TILE;
            const int i_end = min(T, (c + 1) * TILE);
            const int nt = (c + 1) * TILE + tid;
            const double nx = (c + 1 < ntiles && nt < T) ? gx[nt] : 0.0;   // next tile, a whole tile ahead
            const double *xs = sx + (c & 1) * TILE - i_begin;
            for (int i = i_begin; i < i_end; ++i) {
                const double x = xs[i];
                const int slot_prev = slot == 0 ? mv - 1 : slot - 1;      // row i-1
                const int slot_n1 = slot + 1 == mv ? 0 : slot + 1;        // row i+1-mv
                const double *pb = pub + (size_t)(i & 1) * G;
                const int32_t *pbt = ptag + (size_t)(i & 1) * G;
                double *pn = pub + (size_t)((i + 1) & 1) * G;
                int32_t *pnt = ptag + (size_t)((i + 1) & 1) * G;
                for (int g = tid; g < G; g += NT) {
                    const double e = fabs(x - sv[g]) - lam;
                    for (int s = 0; s < mv; ++s)
                        if (s != slot) ring[(size_t)s * G + g] += e;
                    double best = INF;
                    int32_t bt = -1;
                    const double stay = ring[(size_t)slot_prev * G + g];
                    if (stay < best) {
                        best = stay;
                        bt = rtag[(size_t)slot_prev * G + g];
                    }
                    const int e0 = sptr[g], e1 = sptr[g + 1];
                    for (int q = e0; q < e1; ++q) {
                        const int pq = sidx[q];
                        const double cnd = pb[pq] + e;
                        if (cnd < best) {
                            best = cnd;
                            bt = pbt[pq];
                        }
                    }
                    const int fl = sflag[g];
                    if ((fl & 1) && e < best) {                            // a path may start here
                        best = e;
                        bt = i;
                    }
                    ring[(size_t)slot * G + g] = best;
                    rtag[(size_t)slot * G + g] = bt;
                    pn[g] = ring[(size_t)slot_n1 * G + g];
                    pnt[g] = rtag[(size_t)slot_n1 * G + g];
                    if (fl > 1) {                                          // a component's end state: its owner only
                        const int k = (fl >> 1) - 1;
                        if (best < sbest[k]) {
                            sbest[k] = best;
                            slo[k] = bt;
                            shi[k] = i;
                        }
                    }
                }
                slot = slot_n1;
                __syncthreads();
            }
            sx[((c + 1) & 1) * TILE + tid] = nx;
            __syncthreads();
        }
        for (int c = tid; c < C; c += NT) {
            const size_t o = (size_t)m.read * p.n_aut + p.comps[gd.comp0 + c].aut;
            const double b = sbest[c];
            p.score[o] = b;
            p.lo[o] = slo[c];
            p.hi[o] = shi[c];
            p.status[o] = b == INF ? WSTR_LOCATE_NO_PATH : b < 0.0 ? WSTR_LOCATE_FOUND : WSTR_LOCATE_NOT_FOUND;
        }
    }
}

// the rule of assign.choose_loci, per (read, locus)
__global__ void assign_reduce_kernel(const double *__restrict__ score, const int32_t *__restrict__ lo,
                                     const int32_t *__restrict__ hi, const int32_t *__restrict__ status,
                                     int64_t n_pairs, int n_loci, wstr_assign_hit *__restrict__ hits,
                                     int32_t *__restrict__ n_hits) {
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n_pairs; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = k * CHAINS;            // = read * n_aut + locus * CHAINS
        const bool t = status[o] == WSTR_LOCATE_FOUND && status[o + 1] == WSTR_LOCATE_FOUND && hi[o] < lo[o + 1];
        const bool r = status[o + 2] == WSTR_LOCATE_FOUND && status[o + 3] == WSTR_LOCATE_FOUND && hi[o + 2] < lo[o + 3];
        if (!t && !r) continue;
        const int strand = t && r ? (score[o + 2] + score[o + 3] < score[o] + score[o + 1] ? 1 : 0) : (r ? 1 : 0);
        const int64_t a = o + 2 * strand;
        wstr_assign_hit h;
        h.read = (int32_t)(k / n_loci);
        h.locus = (int32_t)(k % n_loci);
        h.strand = strand;
        h.pad_ = 0;
        h.left_lo = lo[a];
        h.left_hi = hi[a];
        h.right_lo = lo[a + 1];
        h.right_hi = hi[a + 1];
        h.left_score = score[a];
        h.right_score = score[a + 1];
        hits[atomicAdd(n_hits, 1)] = h;
    }
}

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct Plan {
    std::vector<GroupDesc> groups;
    std::vector<GroupComp> comps;
    int mv;
    size_t smem, slab;
    size_t o_auts, o_groups, o_comps, o_items, bytes;   // [queue][automata][groups][comps][items]: staged
    int64_t table_off, ring_off, total;           // [table][ring slabs]: written by the kernels
};

// Loci (CHAINS automata each) packed greedily, in order, into groups of at most GROUP_SMEM; a locus that
// does not fit alone is a group of its own with its rings in the workspace.
int make_plan(wstr_automaton *const *automata, int n_aut, int n_reads, int sms, Plan &pl) {
    if (!automata || n_aut <= 0 || n_aut % CHAINS || n_reads < 0) return WSTR_ERR_INVALID_ARGUMENT;
    pl.mv = automata[0] ? automata[0]->dev.mv : 0;
    for (int a = 0; a < n_aut; ++a)
        if (!automata[a] || automata[a]->dev.mv != pl.mv) return WSTR_ERR_INVALID_ARGUMENT;
    const int mv = pl.mv;
    pl.groups.clear();
    pl.comps.clear();
    GroupDesc cur{0, 0, 0, 0, 0, 0};
    auto close = [&]() {
        if (cur.C == 0) return;
        cur.ring_gmem = group_smem(mv, cur.G, cur.E, cur.C, true) > GROUP_SMEM;
        pl.groups.push_back(cur);
        cur = GroupDesc{0, 0, 0, (int32_t)pl.comps.size(), 0, 0};
    };
    for (int l = 0; l < n_aut / CHAINS; ++l) {
        int uG = 0, uE = 0;
        for (int q = 0; q < CHAINS; ++q) {
            uG += automata[l * CHAINS + q]->dev.S;
            uE += automata[l * CHAINS + q]->n_edges;
        }
        if (cur.C > 0 && group_smem(mv, cur.G + uG, cur.E + uE, cur.C + CHAINS, true) > GROUP_SMEM) close();
        for (int q = 0; q < CHAINS; ++q) {
            const wstr_automaton *A = automata[l * CHAINS + q];
            pl.comps.push_back(GroupComp{l * CHAINS + q, cur.G, cur.E, 0});
            cur.G += A->dev.S;
            cur.E += A->n_edges;
            cur.C += 1;
        }
    }
    close();
    pl.smem = 0;
    size_t ring = 0;
    for (const GroupDesc &g : pl.groups) {
        const size_t s = group_smem(mv, g.G, g.E, g.C, !g.ring_gmem);
        if (s > SMEM_MAX) return WSTR_ERR_TOO_MANY_STATES;
        pl.smem = std::max(pl.smem, s);
        if (g.ring_gmem) ring = std::max(ring, ring_bytes(mv, g.G));
    }
    const size_t n_items = (size_t)n_reads * pl.groups.size();
    if (n_items > (size_t)INT32_MAX) return WSTR_ERR_INVALID_ARGUMENT;
    pl.o_auts = 16;
    pl.o_groups = align256(pl.o_auts + sizeof(DevAutomaton) * (size_t)n_aut);
    pl.o_comps = align256(pl.o_groups + sizeof(GroupDesc) * pl.groups.size());
    pl.o_items = align256(pl.o_comps + sizeof(GroupComp) * pl.comps.size());
    pl.bytes = align256(pl.o_items + sizeof(AsgItem) * n_items);
    pl.table_off = (int64_t)pl.bytes;
    pl.slab = align256(ring);
    pl.ring_off = pl.table_off + (int64_t)align256((size_t)n_reads * n_aut * 20);
    const int grid = std::max(1, std::min((int)std::min(n_items, (size_t)INT32_MAX), 2 * sms));
    pl.total = pl.ring_off + (int64_t)(ring ? pl.slab * grid : 0);
    return WSTR_OK;
}

int device_sms(int *sms) {
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    WSTR_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return WSTR_OK;
}

}  // namespace

extern "C" int64_t wstr_assign_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata, int32_t n_reads) {
    int sms = 0;
    int rc = device_sms(&sms);
    if (rc != WSTR_OK) return rc;
    Plan pl;
    rc = make_plan(automata, n_automata, n_reads, sms, pl);
    return rc != WSTR_OK ? rc : pl.total;
}

extern "C" int wstr_assign_batch(wstr_automaton *const *automata, int32_t n_automata, const double *d_signal,
                                 const int64_t *sig_off, const int32_t *lengths, int32_t n_reads, double offset,
                                 void *d_table, wstr_assign_hit *d_hits, int32_t *d_n_hits, void *d_workspace,
                                 int64_t workspace_bytes, void *stream) {
    if (!sig_off || !lengths || n_reads < 0 || !(offset == offset)) return WSTR_ERR_INVALID_ARGUMENT;
    if (!d_hits || !d_n_hits || (reinterpret_cast<uintptr_t>(d_table) & 7)) return WSTR_ERR_INVALID_ARGUMENT;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (n_reads == 0) {
        WSTR_CUDA(cudaMemsetAsync(d_n_hits, 0, sizeof(int32_t), s));
        return WSTR_OK;
    }
    if (!d_signal || !d_workspace || (reinterpret_cast<uintptr_t>(d_workspace) & 15)) return WSTR_ERR_INVALID_ARGUMENT;
    for (int r = 0; r < n_reads; ++r)
        if (lengths[r] < 0 || lengths[r] > WSTR_LOCATE_MAX_SAMPLES || sig_off[r] < 0) return WSTR_ERR_INVALID_ARGUMENT;
    int sms = 0;
    int rc = device_sms(&sms);
    if (rc != WSTR_OK) return rc;
    Plan pl;
    rc = make_plan(automata, n_automata, n_reads, sms, pl);
    if (rc != WSTR_OK) return rc;
    if (workspace_bytes < pl.total) return WSTR_ERR_WORKSPACE_TOO_SMALL;

    const int n_groups = (int)pl.groups.size();
    void *h = nullptr, *token = nullptr;
    rc = wstr_stage_begin(pl.bytes, &h, &token);
    if (rc != WSTR_OK) return rc;
    unsigned char *block = static_cast<unsigned char *>(h);
    *reinterpret_cast<int32_t *>(block) = 0;                                   // the work counter
    DevAutomaton *ha = reinterpret_cast<DevAutomaton *>(block + pl.o_auts);
    for (int a = 0; a < n_automata; ++a) ha[a] = automata[a]->dev;
    std::copy(pl.groups.begin(), pl.groups.end(), reinterpret_cast<GroupDesc *>(block + pl.o_groups));
    std::copy(pl.comps.begin(), pl.comps.end(), reinterpret_cast<GroupComp *>(block + pl.o_comps));
    AsgItem *hi = reinterpret_cast<AsgItem *>(block + pl.o_items);
    std::vector<int> idx(n_reads);
    for (int r = 0; r < n_reads; ++r) idx[r] = r;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return lengths[a] > lengths[b]; });
    size_t k = 0;
    for (int q = 0; q < n_reads; ++q)
        for (int g = 0; g < n_groups; ++g, ++k) {      // a read's groups one after the other: the read stays in L2
            const int r = idx[q];
            hi[k].sig_off = sig_off[r];
            hi[k].T = lengths[r];
            hi[k].read = r;
            hi[k].group = g;
            hi[k].pad_ = 0;
        }
    unsigned char *ws = static_cast<unsigned char *>(d_workspace);
    rc = wstr_stage_commit(token, ws, pl.bytes, s);
    if (rc != WSTR_OK) return rc;

    static unsigned long long attr_done = 0ull;      // devices the function attributes are set on
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    if (!((attr_done >> (dev & 63)) & 1ull)) {
        WSTR_CUDA(cudaFuncSetAttribute(locate_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));
        WSTR_CUDA(cudaFuncSetAttribute(locate_group_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
        attr_done |= 1ull << (dev & 63);
    }
    int per_sm = 1;
    WSTR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, locate_group_kernel, NT, pl.smem));
    per_sm = std::max(1, std::min(per_sm, 2));        // the ring slabs are sized for two CTAs per SM
    const int n_items = (int)k;
    const int grid = std::min(n_items, sms * per_sm);
    const size_t m = (size_t)n_reads * n_automata;
    unsigned char *tab = d_table ? static_cast<unsigned char *>(d_table) : ws + pl.table_off;
    AsgParams p;
    p.auts = reinterpret_cast<const DevAutomaton *>(ws + pl.o_auts);
    p.groups = reinterpret_cast<const GroupDesc *>(ws + pl.o_groups);
    p.comps = reinterpret_cast<const GroupComp *>(ws + pl.o_comps);
    p.items = reinterpret_cast<const AsgItem *>(ws + pl.o_items);
    p.n = n_items;
    p.n_aut = n_automata;
    p.queue = reinterpret_cast<int32_t *>(ws);
    p.signal = d_signal;
    p.offset = offset;
    p.score = reinterpret_cast<double *>(tab);
    p.lo = reinterpret_cast<int32_t *>(tab + 8 * m);
    p.hi = p.lo + m;
    p.status = p.hi + m;
    p.ring_gmem = ws + pl.ring_off;
    p.ring_slab = (int64_t)pl.slab;
    wstr_prof_begin(0, s);
    locate_group_kernel<<<grid, NT, pl.smem, s>>>(p, pl.mv);
    WSTR_CUDA(cudaGetLastError());
    WSTR_CUDA(cudaMemsetAsync(d_n_hits, 0, sizeof(int32_t), s));
    const int64_t pairs = (int64_t)n_reads * (n_automata / CHAINS);
    const int rgrid = (int)std::min<int64_t>((pairs + 255) / 256, (int64_t)sms * 8);
    assign_reduce_kernel<<<rgrid, 256, 0, s>>>(p.score, p.lo, p.hi, p.status, pairs, n_automata / CHAINS, d_hits,
                                               d_n_hits);
    wstr_prof_end(s);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}
