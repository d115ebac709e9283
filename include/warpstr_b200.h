/* warpstr_b200 -- C ABI of the B200-native WarpSTR caller hot path.
 *
 * The reference (fmfi-compbio/warpstr) is pure Python and has no FFI of its own; each
 * entry point below names the reference interface it replaces (file:line relative to the
 * reference tree).  INTEGRATION.md shows the ctypes stubs a WarpSTR maintainer would add
 * to src/caller/wrapper.py to call them.
 *
 * Conventions
 *   - every function returns 0 (WSTR_OK) or a negative WSTR_ERR_* code, never throws;
 *   - "d_" pointers are CUDA device pointers on the current device (e.g. taken from
 *     torch.Tensor.data_ptr()); all other pointers are host pointers and are consumed
 *     before the call returns;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); all device work
 *     is enqueued on it and the call returns without synchronising unless stated;
 *   - per-read problems are reported in d_status[read] (WSTR_READ_*), the batch goes on.
 */
#ifndef WARPSTR_B200_H
#define WARPSTR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WSTR_OK 0
#define WSTR_ERR_INVALID_ARGUMENT (-1)
#define WSTR_ERR_CUDA (-2)
#define WSTR_ERR_TOO_MANY_STATES (-3)     /* states x min_values_per_state beyond the catch-all kernel's shared memory (~20 000) */
#define WSTR_ERR_UNSUPPORTED (-4)         /* e.g. a state with more than 254 incoming edges */
#define WSTR_ERR_WORKSPACE_TOO_SMALL (-5)
#define WSTR_ERR_NO_DEVICE (-6)

/* d_status values */
#define WSTR_READ_OK 0
#define WSTR_READ_TOO_SHORT 1             /* T <= min_values_per_state: reference raises IndexError (caller.py:206-208) */
#define WSTR_READ_BACKTRACK 2             /* reference: RuntimeError('Unexpected error during backtracking'), caller.py:290-291 */
#define WSTR_READ_NO_REPEAT_STATE 3       /* reference: IndexError from trues[0], caller.py:383-384 */
#define WSTR_READ_SPLINE 4                /* reference: FITPACK error / too few points, caller.py:311 */
#define WSTR_READ_SPLINE_KNOTS 5          /* smoothing spline needs interior knots: evaluate this read on the host */
#define WSTR_READ_SEGMENT 6               /* reference: IndexError inside mask_bad_repeats, caller.py:336,358-361,393-411 */

typedef struct wstr_automaton wstr_automaton;

/* ---- library ------------------------------------------------------------------------- */
int wstr_version(void);
const char *wstr_error_string(int code);
/* last CUDA error text seen by this thread (empty string if none) */
const char *wstr_last_cuda_error(void);

/* ---- (1) expected-signal generation -------------------------------------------------------
 * Replaces PoreModel.get_value (src/squiggler/pore_model.py:45-47) applied to every sliding
 * k-mer of a sequence, i.e. Squiggler._generate_signal (src/squiggler/Squiggler.py:20-28).
 * d_seq: n ASCII bases; d_table: 4^k normalised levels in lexicographic ACGT order;
 * d_out: n-k+1 levels.  *d_bad is incremented for every k-mer containing a non-ACGT base
 * (its output is NaN); the reference raises IndexError for such a k-mer. */
int wstr_pore_lookup(const uint8_t *d_seq, int64_t n, const double *d_table, int32_t k,
                     double *d_out, int32_t *d_bad, void *stream);

/* ---- (2) per-read normalisation -----------------------------------------------------------
 * Replaces Fast5.get_data_processed (src/schemas/fast5.py:45-57): whole-read spike removal
 * (brute_remove :90-101, or medfilt 3/5 :72-75, or none) followed by normalize_signal_mad
 * (:104-114) and the [l_start_raw, r_end_raw] slice.
 * d_raw: concatenated int16 reads, read r = d_raw[raw_off[r] .. raw_off[r+1]);
 * spike_mode: 0 None, 1 Brute, 3 median3, 5 median5;
 * window [win_lo[r], win_hi[r]] (inclusive, as in the reference) is written to
 * d_out + out_off[r] as float64.  d_shift_scale (optional, may be NULL) receives
 * {shift, scale} per read.  d_workspace: wstr_normalize_workspace_bytes(n_reads) bytes.
 * The samples are fetched in whole 16-byte words: if d_raw's first or last sample is not 16-byte
 * aligned, up to 14 bytes in front of / behind the buffer are read (and ignored) -- inside the
 * allocation granule for a cudaMalloc'd or torch buffer. */
int64_t wstr_normalize_workspace_bytes(int32_t n_reads);
int wstr_normalize_batch(const int16_t *d_raw, const int64_t *raw_off, const int32_t *win_lo,
                         const int32_t *win_hi, int32_t n_reads, int32_t spike_mode,
                         double *d_out, const int64_t *out_off, double *d_shift_scale,
                         void *d_workspace, int64_t workspace_bytes, void *stream);

/* ---- (2b) reads that are already normalised, shipped compactly -----------------------------------
 * Fast5.get_data_processed ends with `(data - shift) / scale` on the spike-filtered int16 samples
 * (src/schemas/fast5.py:113); a caller that holds those int16 window samples and the read's
 * {shift, scale} (e.g. from wstr_normalize_batch's d_shift_scale) can hand them over instead of the
 * float64 window -- 2 instead of 8 bytes per sample across PCIe -- and gets the same bits:
 * d_out[out_off[r] + t] = ((double)d_raw[raw_off[r] + t] - shift_r) / scale_r, t < lengths[r].
 * d_shift_scale: device, {shift, scale} per read.  Reads whose raw_off is a multiple of 8 and out_off
 * even take the vector path. */
int64_t wstr_dequantize_workspace_bytes(int32_t n_reads);
int wstr_dequantize_batch(const int16_t *d_raw, const int64_t *raw_off, const int32_t *lengths,
                          const double *d_shift_scale, int32_t n_reads, double *d_out,
                          const int64_t *out_off, void *d_workspace, int64_t workspace_bytes, void *stream);

/* ---- (2c) VBZ-compressed raw signal --------------------------------------------------------------
 * Replaces the StreamVByte + zig-zag delta half of the VBZ HDF5 filter (nanoporetech/vbz_compression)
 * that h5py runs when the reference reads Raw/.../Signal (src/schemas/fast5.py:50-52); zstd stays on the
 * host.  Chunk c's body after zstd is d_payload[in_off[c] .. in_off[c] + in_bytes[c]); kind[c]:
 *   WSTR_VBZ_KIND_V0   VBZ version 0: ceil(n/4) bytes of 2-bit codes (c + 1 data bytes), then the data;
 *   WSTR_VBZ_KIND_V1   VBZ version 1 (16-bit integers): ceil(n/8) bytes of 1-bit keys, then the data;
 *   WSTR_VBZ_KIND_RAW  verbatim little-endian int16 (a chunk the host decoded itself).
 * n_samples[c] is the count the body codes (the VBZ header's size / 2); the first n_out[c] <= n_samples[c]
 * samples are written to d_raw + out_off[c] (HDF5's last chunk of a dataset codes a whole chunk).
 * zigzag[c] != 0: the values are zig-zag deltas, summed from 0 in every chunk.  Bit-exact with
 * warpstr_b200/fast5.py:vbz_decompress including its wrap-around to 16 bits; its format errors become
 * d_status[c] (WSTR_VBZ_*), and a bad chunk leaves its own output range undefined and nothing else.
 * The payload is fetched in whole 16-byte words: d_payload and every in_off must be 16-byte aligned, and
 * the bytes up to in_off + in_bytes rounded up to 16 readable (the Python layer pads each chunk with
 * zeros); no byte outside that padded span is read.  Output ranges of the chunks must not overlap.
 * d_workspace: wstr_vbz_workspace_bytes(n_chunks) bytes; the chunk table travels through the staging
 * slot like every other call's host arrays. */
#define WSTR_VBZ_KIND_V0 0
#define WSTR_VBZ_KIND_V1 1
#define WSTR_VBZ_KIND_RAW 2
#define WSTR_VBZ_OK 0
#define WSTR_VBZ_TRUNCATED_CONTROL 1      /* fewer payload bytes than the control (v0) or key (v1) block */
#define WSTR_VBZ_SHORT_DATA 2             /* v0: the data block is shorter than the codes need (extra bytes are fine) */
#define WSTR_VBZ_LENGTH_MISMATCH 3        /* v1: the data block is not exactly as long as the keys say */
int64_t wstr_vbz_workspace_bytes(int32_t n_chunks);
int wstr_vbz_decode_batch(const uint8_t *d_payload, const int64_t *in_off, const int64_t *in_bytes,
                          const int32_t *n_samples, const int32_t *n_out, const int32_t *kind,
                          const int32_t *zigzag, const int64_t *out_off, int32_t n_chunks, int16_t *d_raw,
                          int32_t *d_status, void *d_workspace, int64_t workspace_bytes, void *stream);

/* ---- (3) DTW state automaton ----------------------------------------------------------------
 * wstr_automaton_create uploads one strand's automaton: the flat form of StateAutomata
 * (src/caller/automata.py:36-48).  All arrays are host pointers.
 *   values[S]   State.value             seq_idx[S]  State.seq_idx
 *   in_ptr[S+1], in_idx[E]              CSR of State.incoming, order preserved
 *   rep_mask[S] StateAutomata.mask      last_base[S] last character of State.kmer
 *   endstate    StateAutomata.endstate  flank_length Locus.flank_length
 *   min_values_per_state                tr_calling_config.min_values_per_state: any value > 1, as in
 *                                       the reference (src/config.py:115).  Automata and settings the
 *                                       register-resident kernels are built for (up to 512 states, in-degree
 *                                       <= 4, min_values_per_state 2..8) run on those; everything else on the
 *                                       catch-all kernel, same results.
 */
int wstr_automaton_create(const double *values, const int32_t *seq_idx, const int32_t *in_ptr,
                          const int32_t *in_idx, const uint8_t *rep_mask, const uint8_t *last_base,
                          int32_t n_states, int32_t endstate, int32_t flank_length,
                          int32_t min_values_per_state, wstr_automaton **out);
int wstr_automaton_destroy(wstr_automaton *a);
/* Testing aid: when on, automata created afterwards use the catch-all kernel even where a
 * specialised layout exists (the two must agree bit for bit). */
int wstr_set_generic_only(int32_t on);
/* Host-only dry run of the kernel layout (no device needed): info[0]=chain slots per lane (KC),
 * info[1]=generic slots per lane (KG), info[2]=candidates the generic slots are unrolled for (2 or 4;
 * 100+d: one for every generic slot but the last, d for the last),
 * info[3]=lanes holding chains, info[4]=states placed in generic slots; state_of_pos (optional)
 * receives the state at each of the 32*(KC+KG) positions, -1 = padding.  All zero: no specialised
 * layout, the automaton runs on the catch-all kernel. */
int wstr_automaton_plan(const int32_t *in_ptr, const int32_t *in_idx, int32_t n_states,
                        int32_t min_values_per_state, int32_t *info, int32_t *state_of_pos, int32_t n_pos);
/* info[0]=states per lane (K), info[1]=direction-code bits per lane per row (32/info[1] rows
 * share a 32-bit word), info[2]=chain slots (KC), info[3]=generic slots (KG), info[4]=n_states,
 * info[5]=n_edges, info[6]=states placed in generic slots, info[7]=1 if no edge leads from a
 * state kept by the end band into a skipped one (the band test then stops mv rows into it),
 * info[8]=candidate encoding of the generic slots (DEG: 2 or 4 per slot, 100 + d "low", 200 + 10a + b
 * "graded"; 0 for the catch-all kernel).  Copies min(n_info, 9) values. */
int wstr_automaton_info(const wstr_automaton *a, int32_t *info, int32_t n_info);
/* state index stored at each of the 32*K kernel positions (-1 = padding); for tests */
int wstr_automaton_layout(const wstr_automaton *a, int32_t *state_of_pos, int32_t n_pos);

/* Bytes of device workspace wstr_warp_batch / wstr_call_batch need to process all reads in
 * one wave.  A smaller workspace is legal (>= the value returned for the single largest read
 * plus metadata): the batch is then processed in several waves.
 * Both calls are asynchronous with respect to the host: the per-call plan (read records,
 * processing order) is written into pinned mapped memory and copied in by a kernel on `stream`;
 * no cudaMemcpy/cudaMemset is issued, so the copy engines stay free for the caller's own
 * transfers.  A process may drive several devices: every call works on the current device (the one its
 * automata were created on and its pointers belong to). */
int64_t wstr_warp_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                  const int32_t *read_automaton, const int32_t *lengths,
                                  int32_t n_reads);

/* One DP pass + traceback per read.  Replaces WarpSTR.warp (src/caller/caller.py:189-193) =
 * _calc_dtw_astates (:198-245) + _backtracking (:247-301), for a batch.
 *   d_signal     float64 samples; read r = d_signal[sig_off[r] .. sig_off[r]+lengths[r]);
 *                sig_off[r] must be even (16-byte aligned) and the buffer readable one
 *                element past an odd-length read;
 *   d_maskbits   NULL for the first pass, else bit t of read r (bit (t&31) of word
 *                mask_off[r] + (t>>5)) set = badmask[t] (dwell min_values_per_state-1 allowed);
 *   d_trace      int32 state index per sample, same offsets as d_signal (WarpResult.trace);
 *   d_end_cost   optional (NULL ok): D[T-1, endstate] per read;
 *   d_status     int32 per read.
 */
int wstr_warp_batch(wstr_automaton *const *automata, int32_t n_automata,
                    const int32_t *read_automaton, const double *d_signal, const int64_t *sig_off,
                    const int32_t *lengths, const uint32_t *d_maskbits, const int64_t *mask_off,
                    int32_t n_reads, void *d_workspace, int64_t workspace_bytes,
                    int32_t *d_trace, double *d_end_cost, int32_t *d_status, void *stream);

/* ---- (3b) STR window search in whole reads --------------------------------------------------------
 * Replaces the two steps of the reference that give a read its window [l_start_raw, r_end_raw] (Guppy's
 * re-basecall with a move table, and the flank alignment mapped through it): the strand's automaton is
 * searched against the whole normalised read (wstr_normalize_batch with window [0, N-1]) by the caller's
 * DP with the cost |x_t - v_j| - offset, a free start in state 0 and a free end (DESIGN.md section 4.5):
 * no mask (back = min_values_per_state on every row), no end band.  Per read:
 *   d_lo / d_hi  int32: the best window, inclusive, in the read's sample indices (-1 when there is no path);
 *   d_score      float64: its score, the least L[i][endstate] (+inf when there is no path);
 *   d_status     int32, WSTR_LOCATE_*: found iff the score is below zero.
 * Bit-exact with oracle/locate_oracle.c:wso_locate.  d_signal / sig_off / lengths as for wstr_warp_batch;
 * lengths up to WSTR_LOCATE_MAX_SAMPLES.  All automata of a call have the same min_values_per_state; any
 * automaton wstr_automaton_create accepts is covered (rings beyond shared memory go to the workspace).
 * d_workspace: wstr_locate_workspace_bytes(...) bytes, 16-byte aligned; the plan travels through the
 * staging slot, nothing is copied by the DMA engines and the call does not block. */
#define WSTR_LOCATE_FOUND 0
#define WSTR_LOCATE_NOT_FOUND 1           /* the best window's score is >= 0: nothing in the read matches */
#define WSTR_LOCATE_NO_PATH 2             /* the read is shorter than the automaton's shortest path */
#define WSTR_LOCATE_MAX_SAMPLES 2147479552 /* 2^31 - 4096 */
int64_t wstr_locate_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata, int32_t n_reads);
int wstr_locate_batch(wstr_automaton *const *automata, int32_t n_automata, const int32_t *read_automaton,
                      const double *d_signal, const int64_t *sig_off, const int32_t *lengths, int32_t n_reads,
                      double offset, int32_t *d_lo, int32_t *d_hi, double *d_score, int32_t *d_status,
                      void *d_workspace, int64_t workspace_bytes, void *stream);

/* ---- whole per-read call --------------------------------------------------------------------------
 * Replaces WarpSTR.run (src/caller/caller.py:117-149) for a batch: first pass, per-run statistics
 * and spline rescale, bad-repeat mask, second pass on the rescaled signal, state-wise costs and
 * decoded sequences -- everything between CallerWrapper.run receiving the workload
 * (src/caller/wrapper.py:104-120) and CallerResult.  Device-resident from the signal in to the
 * per-read results out.
 */
typedef struct {
    int32_t min_values_per_state;   /* tr_calling_config.min_values_per_state (= the automata's) */
    int32_t states_in_segment;      /* tr_calling_config.states_in_segment */
    double threshold;               /* rescaling.threshold */
    double max_std;                 /* rescaling.max_std */
    int32_t method;                 /* rescaling.method: 0 mean, 1 median */
    int32_t reps_as_one;            /* rescaling.reps_as_one (caller.py:69-79) */
    int64_t ttest_guard_ulps;       /* width of the d_ttest_ties test in units in the last place; 0 = 16 */
} wstr_call_params;

typedef struct {
    int32_t *d_len1;        /* len(CallerResult.seq)       -> overview column 'orig'    */
    int32_t *d_len2;        /* len(CallerResult.resc_seq)  -> overview column 'results' */
    double *d_cost1;        /* CallerResult.cost           -> 'dtw_cost1' */
    double *d_cost2;        /* CallerResult.resc_cost      -> 'dtw_cost2' */
    int32_t *d_status;      /* WSTR_READ_* per read */
    uint8_t *d_seq1;        /* optional (NULL ok): CallerResult.seq characters, read r at seq_off[r] */
    uint8_t *d_seq2;        /* optional: CallerResult.resc_seq characters */
    const int64_t *seq_off; /* host; byte offsets, capacity per read >= lengths[r]/(mv-1) + 16 */
    int32_t *d_trace1;      /* optional: first-pass trace, same offsets as the signal */
    int32_t *d_trace2;      /* optional: second-pass trace */
    double *d_rescaled;     /* optional: rescaled signal, same offsets as the signal */
    int32_t *d_ttest_ties;  /* optional: per read, the number of t-test decisions of mask_bad_repeats
                             * (caller.py:347-378) within 16 ulp of flipping.  The reference squares with
                             * libm's pow (np.float64 ** 2), which may differ from x*x in the last bit; a read
                             * with 0 ties is decided identically whatever the libm, a read with ties > 0 should
                             * be re-evaluated where the reference's libm is (the Python layer does). */
} wstr_call_outputs;

/* workspace for processing the whole batch in one wave; anything >= the size for the largest
 * single read works (more waves) */
int64_t wstr_call_workspace_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                  const int32_t *read_automaton, const int32_t *lengths,
                                  int32_t n_reads);
/* The smallest workspace wstr_call_batch accepts for this batch: everything that is per batch (rescaled
 * signal, traces, masks, mid-stage scratch: ~35 B per sample) plus the direction codes of its longest
 * read.  A caller whose memory cannot hold that cuts the batch into several calls. */
int64_t wstr_call_workspace_min_bytes(wstr_automaton *const *automata, int32_t n_automata,
                                      const int32_t *read_automaton, const int32_t *lengths,
                                      int32_t n_reads);
/* read_reverse[r] != 0: the read is on the reverse strand (its sequence is reverse-complemented,
 * caller.py:187).  Other arguments as for wstr_warp_batch. */
int wstr_call_batch(wstr_automaton *const *automata, int32_t n_automata,
                    const int32_t *read_automaton, const uint8_t *read_reverse,
                    const double *d_signal, const int64_t *sig_off, const int32_t *lengths,
                    int32_t n_reads, const wstr_call_params *params, void *d_workspace,
                    int64_t workspace_bytes, const wstr_call_outputs *out, void *stream);

/* ---- kernel timing ------------------------------------------------------------------------------
 * When enabled, every kernel launch of this library is bracketed by CUDA events on the launching
 * stream.  wstr_profile_read waits for them and returns, per category (0 DP fill + traceback,
 * 1 mid-stage, 2 normalisation, 3 pore lookup, 4 upload of the per-call host plan), the summed
 * device time in ms and the number of launches since the last read. */
int wstr_profile_enable(int32_t on);
int wstr_profile_read(double *ms, int32_t *launches, int32_t n_categories);

/* ---- measurement helper ---------------------------------------------------------------------
 * Times a dependent-free stream of FP64 adds on every SM (the pipe the DP is bound by) and
 * returns the achieved rate in 1e12 DADD/s (lane operations); used by bench.py as the
 * measured roofline denominator.  Synchronises. */
int wstr_measure_fp64_add_rate(double *tera_adds_per_s, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WARPSTR_B200_H */
