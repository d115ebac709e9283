"""GPU: the stage between the two DP passes (csrc/midstage.cu) against the oracle's mid-stage, on each size
switch of the kernels.  Every read's rescaled signal, costs, lengths, sequences and status are compared
bit for bit with oracle/caller_oracle.py's after_first_pass / after_second_pass applied to the device's
own traces (oracle/bulk.py:run_midstage, no DP on the host).  The bad-repeat mask is not an output of the
call: the device's second pass is replayed with the oracle's mask and must reproduce the device's trace2.
Reads with a t-test decision within rounding distance of flipping (`ties`, decided by the host's libm) are
left out of the bit comparison and counted, as in test_gpu_bulk.py.

Each group asserts, from facts the oracle reports about its reads, that the branch it is there for was
taken, so that a change of the read generator fails the test instead of silently testing less.

WSTR_MIDSTAGE_SCALE scales the read counts that are free to change (default 1; the 16 384-read call
of the fit-kernel group is fixed by the kernel's switch)."""
import dataclasses
import os
from collections import Counter

import numpy as np
import pytest

from warpstr_b200 import synth
from warpstr_b200.automata import StateAutomata
from warpstr_b200.config import CallerConfig, RescalerConfig

pytestmark = pytest.mark.gpu

SCALE = float(os.environ.get('WSTR_MIDSTAGE_SCALE', '1'))
F = 110
PIPE_MAX_READS = 16384          # FIT_PIPE_MAX_READS in midstage.cu


def _n(k: int) -> int:
    return max(1, int(round(k * SCALE)))


def _reads(locus, n, seed, noise=0.15, dwell=(5, 13)):
    """(signals, reverse flags) of ``n`` synthetic reads of ``locus``."""
    sig, off, ln, rev, _ = synth.make_read_batch(locus, n, seed=seed, noise=noise, dwell=dwell)
    return [sig[o:o + k].copy() for o, k in zip(off, ln)], rev.astype(bool)


def _quantised(signals, seed):
    """The reads on the grid the int16 routes produce: DAC counts (the inverse of the normalisation
    synth.to_raw_int16 uses) mapped back through a shift and scale of each read's own."""
    rng = np.random.default_rng(seed)
    out = []
    for s in signals:
        shift = 90.8717 * 5.85 + rng.uniform(-0.5, 0.5)
        scale = 9.8354 * 5.85 * (1.0 + rng.uniform(-0.01, 0.01))
        out.append((np.rint((90.8717 + 9.8354 * s) * 5.85) - shift) / scale)
    return out


def _c9(units, seed):
    """A (GGGGCC) locus whose allele has ``units`` = (lo, hi) repeat units."""
    loc = synth.make_locus(f'C9_{units[0]}_{units[1]}', seed=seed, recipe='C9ORF72_100')
    return dataclasses.replace(loc, units=(('GGGGCC',) + tuple(units),))


class Setup:
    """An engine with both strands of each locus (automaton 2 i + reverse) and the oracle's view of it."""

    def __init__(self, loci, cc=None, rc=None):
        from warpstr_b200.caller import CallerEngine
        self.cc, self.rc = cc or CallerConfig(), rc or RescalerConfig()
        self.eng = CallerEngine(self.cc, self.rc)
        self.regexes = [rx for loc in loci for rx in (loc.template_regex, loc.reverse_regex)]
        for rx in self.regexes:
            self.eng.add_automaton(StateAutomata(rx), F)
        self.knobs = (self.cc.min_values_per_state, self.cc.states_in_segment, self.rc.reps_as_one,
                      self.rc.threshold, self.rc.max_std, self.rc.method)


class Call:
    """One call_packed with the debug outputs, on host, and the mid-stage fit kernels it launched."""

    def __init__(self, st: Setup, signals, aut, rev):
        import torch
        from torch.profiler import ProfilerActivity, profile
        self.signals, self.aut, self.rev = signals, np.asarray(aut, dtype=np.int32), np.asarray(rev, dtype=bool)
        d_sig, self.off, self.lengths, a, r = st.eng.upload(signals, self.aut, self.rev)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            o = st.eng.call_packed(d_sig, self.off, self.lengths, a, r, want_debug=True, allow_split=False)
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages()]
        self.fit_kernels = {k for k in ('mid_fit_pipe_kernel', 'mid_fit_kernel') if any(k in n for n in names)}
        self.g = {k: (v.cpu().numpy() if hasattr(v, 'cpu') else v) for k, v in o.items()}

    def sample(self, key, r):
        a = int(self.off[r])
        return self.g[key][a:a + int(self.lengths[r])]

    def seq(self, key, r):
        a = int(self.g['seq_off'][r])
        return self.g[key][a:a + int(self.g['len' + key[-1]][r])].tobytes().decode()

    def status(self, r):
        return int(self.g['status'][r])


def _compare(label, st: Setup, c: Call, idx=None, min_full=0.9):
    """Device vs the oracle's mid-stage on the device's traces, for reads ``idx`` (default all).  A read with
    t-test ties is compared on what precedes the mask (rescaled signal, first cost, length and sequence);
    every other read on everything, at least a share ``min_full`` of the reads.  Returns the oracle's per-read
    dicts (None for a read whose DP failed on the device: there is no mid-stage to compare)."""
    from oracle import bulk
    idx = np.arange(len(c.signals)) if idx is None else np.asarray(idx)
    dp_ok = [int(r) for r in idx if c.status(r) not in (1, 2)]          # WSTR_READ_TOO_SHORT / _BACKTRACK
    want = bulk.run_midstage(st.regexes, F, [c.signals[r] for r in dp_ok], [c.sample('trace1', r) for r in dp_ok],
                             [c.sample('trace2', r) for r in dp_ok], c.aut[dp_ok], c.rev[dp_ok], st.knobs)
    bad = Counter()
    compared, tie_skipped, replay = [], 0, []
    for r, w in zip(dp_ok, want):
        if w['status'] != 0 or c.status(r) != 0:
            bad['status'] += int(w['status'] != c.status(r))
            continue
        bad['rescaled'] += int(not np.array_equal(c.sample('rescaled', r), w['rescaled']))
        bad['cost'] += int(c.g['cost1'][r] != w['cost1'])
        bad['len'] += int(c.g['len1'][r] != len(w['seq1']))
        bad['seq'] += int(c.seq('seq1', r) != w['seq1'])
        if c.g['ties'][r] > 0:       # the mask, and so the second pass, is the host libm's to decide (d_ttest_ties)
            tie_skipped += 1
            continue
        compared.append(r)
        bad['cost'] += int(c.g['cost2'][r] != w['cost2'])
        bad['len'] += int(c.g['len2'][r] != len(w['seq2']))
        bad['seq'] += int(c.seq('seq2', r) != w['seq2'])
        replay.append(w['mask'])
    # the mask: the second pass again, on the device's rescaled signal with the oracle's mask
    t2 = st.eng.warp_batch([c.sample('rescaled', r) for r in compared], c.aut[compared], replay)
    bad['mask'] += sum(int(not np.array_equal(t, c.sample('trace2', r))) for r, t in zip(compared, t2))
    masked = float(np.mean([m.any() for m in replay])) if replay else 0.0
    errors = Counter(w['error'] for w in want if w['error'])
    print(f'\n[{label}] reads {len(idx)}, compared in full {len(compared)}, mismatches {dict(bad)}, reads with '
          f't-test ties (first pass compared only) {tie_skipped}, oracle exceptions {dict(errors)}, DP failures '
          f'{len(idx) - len(dp_ok)}, non-empty masks {masked:.2f}, fit kernels {sorted(c.fit_kernels)}')
    assert not any(bad.values()), (label, dict(bad))
    assert len(compared) >= min_full * len(idx), (label, len(compared), len(idx))
    # the replay proves something only if the masks have bits (every read of these synthetic loci has some)
    assert not compared or masked >= 0.9, (label, masked)
    out = [None] * len(c.signals)
    for r, w in zip(dp_ok, want):
        out[r] = w
    return out


def _anchor(label, st: Setup, c: Call, idx):
    """The full oracle (DP included) on a few reads: sequences and costs, or the device flags the read."""
    from oracle import bulk
    idx = [int(r) for r in idx]
    want = bulk.run_reads(st.regexes, F, [c.signals[r] for r in idx], c.aut[idx], c.rev[idx], knobs=st.knobs)
    bad = 0
    for r, w in zip(idx, want):
        if w[0] == 'error':
            bad += int(c.status(r) == 0)
        elif c.status(r) != 0:
            bad += 1
        elif c.g['ties'][r] == 0:
            bad += int((c.seq('seq1', r), c.seq('seq2', r), c.g['cost1'][r], c.g['cost2'][r]) != tuple(w))
    print(f'[{label}] full oracle on {len(idx)} reads: {bad} mismatches')
    assert bad == 0, label


def _facts(want, key):
    return [w[key] for w in want if w is not None and w['status'] == 0]


def _run_hist(want):
    hs = _facts(want, 'run_hist')
    h = np.zeros(max(len(x) for x in hs), dtype=np.int64)
    for x in hs:
        h[:len(x)] += x
    return h


def _interleave(seed, *parts):
    """Concatenate (signals, aut, rev) parts and shuffle the reads among each other."""
    sigs = [s for p in parts for s in p[0]]
    aut = np.concatenate([p[1] for p in parts]).astype(np.int32)
    rev = np.concatenate([p[2] for p in parts]).astype(bool)
    order = np.random.default_rng(seed).permutation(len(sigs))
    return [sigs[i] for i in order], aut[order], rev[order]


def _part(st_index, signals, rev):
    return signals, 2 * st_index + rev.astype(np.int32), rev


# ---- A: long runs: pairwise16 (incl. n == 16), pairwise_leaf 17..128, the explicit-stack sum > 128,
#         run_median on long runs --------------------------------------------------------------------------
@pytest.mark.parametrize('method', ['mean', 'median'])
def test_long_runs(built_lib, oracle_c, method):
    loci = [synth.make_locus('HD', seed=410), synth.make_locus('DM2', seed=411)]
    st = Setup(loci, rc=RescalerConfig(method=method))
    parts = [_part(i, *_reads(loc, _n(24), seed=412 + i, dwell=(4, 220))) for i, loc in enumerate(loci)]
    c = Call(st, *_interleave(413, *parts))
    want = _compare(f'A long runs {method}', st, c)
    _anchor(f'A long runs {method}', st, c, range(2))
    h = _run_hist(want)
    buckets = {L: int(h[L]) for L in (8, 15, 16, 17, 128, 129)}
    print(f'[A] runs of length {buckets}, > 200: {int(h[201:].sum())}, longest {len(h) - 1}')
    assert all(v > 0 for v in buckets.values()) and h[201:].sum() > 0, buckets


# ---- B: sort sizes (shared memory <= 512 pairs, tiled above) and tied keys ---------------------------------
@pytest.mark.parametrize('method', ['mean', 'median'])
@pytest.mark.parametrize('form,noise', [('float', 0.15), ('quantised', 0.05), ('quantised', 0.2)])
def test_sort_sizes_and_ties(built_lib, oracle_c, form, noise, method):
    loci = [_c9((45, 75), 420), _c9((280, 320), 421), _c9((950, 1000), 422)]
    st = Setup(loci, rc=RescalerConfig(method=method))
    parts = []
    for i, (loc, n) in enumerate(zip(loci, (_n(360), 6, 4))):
        sigs, rev = _reads(loc, n, seed=423 + i, noise=noise)
        if form == 'quantised':
            sigs = _quantised(sigs, seed=426 + i)
        parts.append(_part(i, sigs, rev))
    c = Call(st, *_interleave(429, *parts))
    label = f'B sort {form} {noise} {method}'
    # on the DAC grid a t statistic often lands within a few ulp of 3 (or of its predecessor), a decision the
    # device leaves to the host's libm: at noise 0.05 most reads have one (their first pass is still compared)
    want = _compare(label, st, c, min_full={'float': 0.9, 'quantised': 0.1 if noise < 0.1 else 0.7}[form])
    _anchor(label, st, c, np.flatnonzero(c.aut < 2)[:3])
    m, ties, zero = np.array(_facts(want, 'm')), np.array(_facts(want, 'ties')), sum(_facts(want, 'zero_sd'))
    above = m > 512
    print(f'[{label}] m in [480, 512]: {int(((m >= 480) & (m <= 512)).sum())}, [513, 560]: '
          f'{int(((m >= 513) & (m <= 560)).sum())}, > 4096: {int((m > 4096).sum())}, max {m.max()}, '
          f'> 512 with m mod 512 in [1, 32]: {int((above & (m % 512 >= 1) & (m % 512 <= 32)).sum())}; '
          f'reads with tied keys: {int((ties > 0).sum())} ({int((ties[above] > 0).sum())} of {int(above.sum())} '
          f'above 512); zero-deviation t-test windows {zero}')
    assert ((m >= 480) & (m <= 512)).sum() >= 10 and ((m >= 513) & (m <= 560)).sum() >= 10
    assert (m > 4096).any() and (above & (m % 512 >= 1) & (m % 512 <= 32)).any()
    if form == 'quantised' and method == 'median':
        assert (ties[above] > 0).mean() > 0.5
    if form == 'quantised' and noise == 0.05:
        assert zero > 0


# ---- C: both fit kernels on the same reads ------------------------------------------------------------------
def test_fit_kernels_agree_on_the_same_reads(built_lib, oracle_c):
    locus = synth.make_locus('HD', seed=430)
    st = Setup([locus])
    sigs, rev = _reads(locus, PIPE_MAX_READS + 1, seed=431)
    aut = rev.astype(np.int32)
    n = PIPE_MAX_READS
    pipe = Call(st, sigs[:n], aut[:n], rev[:n])
    thread = Call(st, sigs, aut, rev)
    rng = np.random.default_rng(432)
    sub = np.sort(rng.choice(n, _n(2000), replace=False))
    short = sigs[n][:90]                        # 2 * run_cap > T: the batch no longer fits the pipelined fit
    small = Call(st, [sigs[r] for r in sub] + [short], np.append(aut[sub], aut[n]), np.append(rev[sub], rev[n]))
    print(f'\n[C] fit kernels: {n} reads {sorted(pipe.fit_kernels)}, {n + 1} reads {sorted(thread.fit_kernels)}, '
          f'{len(sub)} + a {len(short)}-sample read {sorted(small.fit_kernels)}')
    assert pipe.fit_kernels == {'mid_fit_pipe_kernel'}
    assert thread.fit_kernels == {'mid_fit_kernel'} and small.fit_kernels == {'mid_fit_kernel'}

    # bit-identical across the three calls, every shared read
    bad = Counter()
    for other, rows in ((thread, np.arange(n)), (small, sub)):
        for k, r in enumerate(rows):
            j = r if other is thread else k
            bad['status'] += int(pipe.status(r) != other.status(j))
            if pipe.status(r) != 0:
                continue
            bad['rescaled'] += int(not np.array_equal(pipe.sample('rescaled', r), other.sample('rescaled', j)))
            bad['cost'] += int(pipe.g['cost1'][r] != other.g['cost1'][j] or pipe.g['cost2'][r] != other.g['cost2'][j])
            bad['len'] += int(pipe.g['len1'][r] != other.g['len1'][j] or pipe.g['len2'][r] != other.g['len2'][j])
    print(f'[C] pipe vs thread kernel on {n} + {len(sub)} shared reads: mismatches {dict(bad)}')
    assert not any(bad.values()), dict(bad)

    _compare('C thread kernel, oracle sample', st, thread, np.sort(rng.choice(n + 1, _n(1000), replace=False)))
    _anchor('C short read', st, small, [len(sub)] + list(range(3)))

    for mv, kernel in ((3, 'mid_fit_kernel'), (5, 'mid_fit_pipe_kernel')):
        st_mv = Setup([locus], cc=CallerConfig(min_values_per_state=mv))
        c = Call(st_mv, sigs[:_n(1000)], aut[:_n(1000)], rev[:_n(1000)])
        assert c.fit_kernels == {kernel}, (mv, c.fit_kernels)
        _compare(f'C mv {mv}', st_mv, c)


# ---- D: the pipelined fit's packing: eight reads of different m per warp, flagged reads among them, a tail
#         warp -------------------------------------------------------------------------------------------------
def test_pipe_kernel_warp_packing(built_lib, oracle_c):
    loci = [synth.make_locus('HD', seed=440), _c9((300, 300), 441)]
    st = Setup(loci)
    hd = _part(0, *_reads(loci[0], _n(2760), seed=442))
    c9 = _part(1, *_reads(loci[1], _n(200), seed=443))
    n_flat = _n(43)
    flat = ([np.full(4000, 40.0) for _ in range(n_flat)], np.zeros(n_flat, dtype=np.int32), np.zeros(n_flat, dtype=bool))
    sigs, aut, rev = _interleave(444, hd, c9, flat)
    assert len(sigs) % 8 and len(sigs) % 32
    c = Call(st, sigs, aut, rev)
    assert c.fit_kernels == {'mid_fit_pipe_kernel'}, c.fit_kernels
    want = _compare('D pipe packing', st, c)
    flagged = np.array([c.status(r) != 0 for r in range(len(sigs))])
    warps_with_flagged = len({r // 8 for r in np.flatnonzero(flagged)})
    print(f'[D] {len(sigs)} reads, {int(flagged.sum())} flagged before the fit '
          f'({Counter(c.status(r) for r in np.flatnonzero(flagged))}), in {warps_with_flagged} of '
          f'{(len(sigs) + 7) // 8} pipe slots; m of the reads {min(_facts(want, "m"))}..{max(_facts(want, "m"))}')
    assert flagged.sum() >= n_flat and warps_with_flagged >= n_flat // 2

    # the same reads in another order (other neighbours in every warp), and some alone
    perm = np.random.default_rng(445).permutation(len(sigs))
    again = Call(st, [sigs[i] for i in perm], aut[perm], rev[perm])
    rng = np.random.default_rng(446)
    alone_idx = set(rng.choice(np.flatnonzero(~flagged), 24, replace=False).tolist())
    bad = Counter()
    for k, r in enumerate(perm):
        others = [(again, k)]
        if r in alone_idx:
            others.append((Call(st, [sigs[r]], aut[r:r + 1], rev[r:r + 1]), 0))
        for o, j in others:
            bad['status'] += int(c.status(r) != o.status(j))
            if c.status(r) == 0:
                bad['rescaled'] += int(not np.array_equal(c.sample('rescaled', r), o.sample('rescaled', j)))
                bad['cost'] += int(c.g['cost1'][r] != o.g['cost1'][j] or c.g['cost2'][r] != o.g['cost2'][j])
    print(f'[D] permuted batch and {len(alone_idx)} reads alone: mismatches {dict(bad)}')
    assert not any(bad.values()), dict(bad)
    _anchor('D pipe packing', st, c, [r for r in range(len(sigs)) if aut[r] < 2][:3])


# ---- E: reps_as_one across automata of one call (scratch sized by the largest), run_median and select_kth --
@pytest.mark.parametrize('method', ['mean', 'median'])
@pytest.mark.parametrize('form', ['float', 'quantised'])
def test_reps_as_one_across_automata(built_lib, oracle_c, form, method):
    loci = [synth.make_locus('HD', seed=450), synth.make_locus('DM2', seed=451), _c9((100, 100), 452)]
    st = Setup(loci, rc=RescalerConfig(reps_as_one=True, method=method))
    parts = []
    for i, loc in enumerate(loci):
        sigs, rev = _reads(loc, _n(80), seed=453 + i, noise=0.2)
        if form == 'quantised':
            sigs = _quantised(sigs, seed=456 + i)
        parts.append(_part(i, sigs, rev))
    c = Call(st, *_interleave(459, *parts))
    label = f'E reps_as_one {form} {method}'
    want = _compare(label, st, c, min_full=0.9 if form == 'float' else 0.7)
    _anchor(label, st, c, range(3))
    g = np.concatenate(_facts(want, 'groups'))
    kinds = {'<= 48 odd': int(((g <= 48) & (g % 2 == 1)).sum()), '<= 48 even': int(((g <= 48) & (g % 2 == 0)).sum()),
             '> 48 odd': int(((g > 48) & (g % 2 == 1)).sum()), '> 48 even': int(((g > 48) & (g % 2 == 0)).sum())}
    print(f'[{label}] group sizes {kinds}, largest {g.max()}')
    assert all(v > 0 for v in kinds.values()), kinds
