// (3b) STR window search in whole reads (DESIGN.md section 4.5).
//
// The caller's DP (dtw_any.cu) run over the whole normalised read with the cost |x_t - v_j| - offset, a free
// start in state 0 on every row and a free end: no mask (back = mv on every row), no end band, no direction
// codes and no traceback.  Instead of a direction per cell, every partial sum carries the row its path
// started on, so the answer -- the best end row of the end state, its score and its start row -- is known
// when the last row is done.  Bit-exact with oracle/locate_oracle.c:wso_locate.
//
// One CTA of 128 threads per read (a work counter hands out reads, longest first), thread t owns states
// t, t+128, ...  Per state a ring of mv running sums, slot (t mod mv) holding
//     L[t][j] + c_{t+1}(j) + ... + c_{i-1}(j)
// summed left to right, and the start row of each; the sums of rows i-mv+1 of every state are published at
// the end of row i for the skip candidates of row i+1 (double-buffered: one __syncthreads per row).  The
// ring lives in shared memory, or, for automata whose mv x S rings do not fit there, in a slab of the
// workspace per CTA (only its owner thread ever touches a ring entry).
#include <algorithm>
#include <vector>

#include "wstr_internal.h"

namespace {

constexpr int NT = 128;
constexpr int TILE = NT;                 // samples per signal tile: one per thread
constexpr size_t SMEM_MAX = 226 * 1024;  // dynamic shared memory per block: sm_100's 227 KB opt-in, less the static part

struct LocRead {
    int64_t sig_off;
    int32_t T, aut, read, pad_;
};

struct LocParams {
    const DevAutomaton *auts;
    const LocRead *reads;        // longest first
    int32_t n;
    int32_t *queue;              // zero when the plan arrives
    const double *signal;
    double offset;
    int32_t *lo, *hi, *status;
    double *score;
    unsigned char *ring_gmem;    // NULL: rings in shared memory; else a slab of ring_slab bytes per CTA
    int64_t ring_slab;
};

__host__ __device__ inline size_t ring_bytes(int mv, int spad) { return (size_t)mv * spad * (sizeof(double) + sizeof(int32_t)); }
// [ring mv x spad doubles][ring tags mv x spad int32] (when in shared memory) [pub 2 x spad][pub tags 2 x spad]
// [v spad][signal 2 x TILE]
__host__ __device__ inline size_t fixed_bytes(int spad) {
    return 2 * (size_t)spad * (sizeof(double) + sizeof(int32_t)) + sizeof(double) * ((size_t)spad + 2 * TILE);
}

__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }

__global__ void __launch_bounds__(NT) locate_kernel(const LocParams p, const int mv, const int spad_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_next;
    unsigned char *fixed = smem_raw;
    unsigned char *rb = p.ring_gmem ? p.ring_gmem + (size_t)blockIdx.x * p.ring_slab : smem_raw;
    if (!p.ring_gmem) fixed += ring_bytes(mv, spad_max);
    double *ring = reinterpret_cast<double *>(rb);                            // [mv][spad_max]
    int32_t *rtag = reinterpret_cast<int32_t *>(ring + (size_t)mv * spad_max);  // [mv][spad_max]
    double *pub = reinterpret_cast<double *>(fixed);                          // [2][spad_max]
    double *sv = pub + 2 * (size_t)spad_max;
    double *sx = sv + spad_max;                                               // [2][TILE]
    int32_t *ptag = reinterpret_cast<int32_t *>(sx + 2 * TILE);               // [2][spad_max]
    const int tid = threadIdx.x;
    const double INF = dinf();
    const double lam = p.offset;
    int cached_aut = -1;

    for (;;) {
        __syncthreads();       // the previous read is done with shared memory
        if (tid == 0) s_next = atomicAdd(p.queue, 1);
        __syncthreads();
        const int r = s_next;
        if (r >= p.n) break;
        const LocRead m = p.reads[r];
        const DevAutomaton *A = p.auts + m.aut;
        const int T = m.T;
        const int S = A->S;
        const int endstate = A->endstate;
        const int32_t *__restrict__ in_ptr = A->in_ptr;
        const int32_t *__restrict__ in_idx = A->in_idx;
        if (m.aut != cached_aut) {
            for (int j = tid; j < S; j += NT) sv[j] = __ldg(A->values + j);
            cached_aut = m.aut;
        }
        // no row yet: every running sum and both published rows are +inf
        for (int j = tid; j < S; j += NT) {
            for (int s = 0; s < mv; ++s) ring[(size_t)s * spad_max + j] = INF;
            pub[j] = INF;
            pub[spad_max + j] = INF;
        }
        const double *__restrict__ gx = p.signal + m.sig_off;
        const int ntiles = (T + TILE - 1) / TILE;
        sx[tid] = tid < T ? gx[tid] : 0.0;
        __syncthreads();

        double best_e = INF;     // end state's best cell so far (its owner's registers)
        int e_lo = -1, e_hi = -1;
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
                const double *pb = pub + (size_t)(i & 1) * spad_max;
                const int32_t *pbt = ptag + (size_t)(i & 1) * spad_max;
                double *pn = pub + (size_t)((i + 1) & 1) * spad_max;
                int32_t *pnt = ptag + (size_t)((i + 1) & 1) * spad_max;
                for (int j = tid; j < S; j += NT) {
                    const double e = fabs(x - sv[j]) - lam;
                    for (int s = 0; s < mv; ++s)
                        if (s != slot) ring[(size_t)s * spad_max + j] += e;
                    double best = INF;
                    int32_t bt = -1;
                    const double stay = ring[(size_t)slot_prev * spad_max + j];
                    if (stay < best) {
                        best = stay;
                        bt = rtag[(size_t)slot_prev * spad_max + j];
                    }
                    const int e0 = __ldg(in_ptr + j), e1 = __ldg(in_ptr + j + 1);
                    for (int q = e0; q < e1; ++q) {
                        const int pq = __ldg(in_idx + q);
                        const double cnd = pb[pq] + e;
                        if (cnd < best) {
                            best = cnd;
                            bt = pbt[pq];
                        }
                    }
                    if (j == 0 && e < best) {                              // a path may start here
                        best = e;
                        bt = i;
                    }
                    ring[(size_t)slot * spad_max + j] = best;
                    rtag[(size_t)slot * spad_max + j] = bt;
                    pn[j] = ring[(size_t)slot_n1 * spad_max + j];
                    pnt[j] = rtag[(size_t)slot_n1 * spad_max + j];
                    if (j == endstate && best < best_e) {
                        best_e = best;
                        e_lo = bt;
                        e_hi = i;
                    }
                }
                slot = slot_n1;
                __syncthreads();
            }
            sx[((c + 1) & 1) * TILE + tid] = nx;
            __syncthreads();
        }
        if (tid == endstate % NT) {
            const int rd = m.read;
            p.score[rd] = best_e;
            p.lo[rd] = e_lo;
            p.hi[rd] = e_hi;
            p.status[rd] = best_e == INF ? WSTR_LOCATE_NO_PATH : best_e < 0.0 ? WSTR_LOCATE_FOUND : WSTR_LOCATE_NOT_FOUND;
        }
    }
}

struct Plan {
    size_t o_auts, o_reads, bytes;    // [queue][DevAutomaton x A][LocRead x n]
    int spad_max, mv;
    bool ring_in_gmem;
    size_t smem, slab;
    int64_t ring_off, ring_bytes_total, total;
};

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

int device_sms(int *sms) {
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    WSTR_CUDA(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return WSTR_OK;
}

int make_plan(wstr_automaton *const *automata, int n_automata, int n_reads, int sms, Plan &pl) {
    if (!automata || n_automata <= 0 || n_reads < 0) return WSTR_ERR_INVALID_ARGUMENT;
    pl.mv = automata[0] ? automata[0]->dev.mv : 0;
    pl.spad_max = 0;
    for (int a = 0; a < n_automata; ++a) {
        if (!automata[a] || automata[a]->dev.mv != pl.mv) return WSTR_ERR_INVALID_ARGUMENT;
        pl.spad_max = std::max(pl.spad_max, (int)automata[a]->dev.spad);
    }
    pl.o_auts = 16;
    pl.o_reads = align256(pl.o_auts + sizeof(DevAutomaton) * (size_t)n_automata);
    pl.bytes = align256(pl.o_reads + sizeof(LocRead) * (size_t)n_reads);
    const size_t fixed = fixed_bytes(pl.spad_max) + 16;
    const size_t ring = ring_bytes(pl.mv, pl.spad_max);
    if (fixed > SMEM_MAX) return WSTR_ERR_TOO_MANY_STATES;
    pl.ring_in_gmem = fixed + ring > SMEM_MAX;
    pl.smem = pl.ring_in_gmem ? fixed : fixed + ring;
    pl.slab = align256(ring);
    const int grid = std::max(1, std::min(n_reads, sms));   // the global-ring form runs one CTA per SM
    pl.ring_off = (int64_t)pl.bytes;
    pl.ring_bytes_total = pl.ring_in_gmem ? (int64_t)(pl.slab * grid) : 0;
    pl.total = pl.ring_off + pl.ring_bytes_total;
    return WSTR_OK;
}

}  // namespace

extern "C" int64_t wstr_locate_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata, int32_t n_reads) {
    int sms = 0;
    int rc = device_sms(&sms);
    if (rc != WSTR_OK) return rc;
    Plan pl;
    rc = make_plan(automata, n_automata, n_reads, sms, pl);
    return rc != WSTR_OK ? rc : pl.total;
}

extern "C" int wstr_locate_batch(wstr_automaton *const *automata, int32_t n_automata, const int32_t *read_automaton,
                                 const double *d_signal, const int64_t *sig_off, const int32_t *lengths,
                                 int32_t n_reads, double offset, int32_t *d_lo, int32_t *d_hi, double *d_score,
                                 int32_t *d_status, void *d_workspace, int64_t workspace_bytes, void *stream) {
    if (!read_automaton || !sig_off || !lengths || n_reads < 0 || !(offset == offset)) return WSTR_ERR_INVALID_ARGUMENT;
    if (n_reads == 0) return WSTR_OK;
    if (!d_signal || !d_lo || !d_hi || !d_score || !d_status || !d_workspace ||
        (reinterpret_cast<uintptr_t>(d_workspace) & 15))
        return WSTR_ERR_INVALID_ARGUMENT;
    for (int r = 0; r < n_reads; ++r)
        if (read_automaton[r] < 0 || read_automaton[r] >= n_automata || lengths[r] < 0 ||
            lengths[r] > WSTR_LOCATE_MAX_SAMPLES || sig_off[r] < 0)
            return WSTR_ERR_INVALID_ARGUMENT;
    int sms = 0;
    int rc = device_sms(&sms);
    if (rc != WSTR_OK) return rc;
    Plan pl;
    rc = make_plan(automata, n_automata, n_reads, sms, pl);
    if (rc != WSTR_OK) return rc;
    if (workspace_bytes < pl.total) return WSTR_ERR_WORKSPACE_TOO_SMALL;

    cudaStream_t s = static_cast<cudaStream_t>(stream);
    void *h = nullptr, *token = nullptr;
    rc = wstr_stage_begin(pl.bytes, &h, &token);
    if (rc != WSTR_OK) return rc;
    unsigned char *block = static_cast<unsigned char *>(h);
    *reinterpret_cast<int32_t *>(block) = 0;                                   // the work counter
    DevAutomaton *ha = reinterpret_cast<DevAutomaton *>(block + pl.o_auts);
    for (int a = 0; a < n_automata; ++a) ha[a] = automata[a]->dev;
    LocRead *hr = reinterpret_cast<LocRead *>(block + pl.o_reads);
    std::vector<int> idx(n_reads);
    for (int r = 0; r < n_reads; ++r) idx[r] = r;
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return lengths[a] > lengths[b]; });
    for (int k = 0; k < n_reads; ++k) {
        const int r = idx[k];
        hr[k].sig_off = sig_off[r];
        hr[k].T = lengths[r];
        hr[k].aut = read_automaton[r];
        hr[k].read = r;
        hr[k].pad_ = 0;
    }
    unsigned char *ws = static_cast<unsigned char *>(d_workspace);
    rc = wstr_stage_commit(token, ws, pl.bytes, s);
    if (rc != WSTR_OK) return rc;

    static unsigned long long attr_done = 0ull;      // devices the function attributes are set on
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    if (!((attr_done >> (dev & 63)) & 1ull)) {
        WSTR_CUDA(cudaFuncSetAttribute(locate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));
        WSTR_CUDA(cudaFuncSetAttribute(locate_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       cudaSharedmemCarveoutMaxShared));
        attr_done |= 1ull << (dev & 63);
    }
    int per_sm = 1;
    if (!pl.ring_in_gmem) {
        WSTR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, locate_kernel, NT, pl.smem));
        if (per_sm < 1) per_sm = 1;
    }
    const int grid = std::min(n_reads, sms * per_sm);
    LocParams p;
    p.auts = reinterpret_cast<const DevAutomaton *>(ws + pl.o_auts);
    p.reads = reinterpret_cast<const LocRead *>(ws + pl.o_reads);
    p.n = n_reads;
    p.queue = reinterpret_cast<int32_t *>(ws);
    p.signal = d_signal;
    p.offset = offset;
    p.lo = d_lo;
    p.hi = d_hi;
    p.status = d_status;
    p.score = d_score;
    p.ring_gmem = pl.ring_in_gmem ? ws + pl.ring_off : nullptr;
    p.ring_slab = (int64_t)pl.slab;
    wstr_prof_begin(0, s);
    locate_kernel<<<grid, NT, pl.smem, s>>>(p, pl.mv, pl.spad_max);
    wstr_prof_end(s);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}
