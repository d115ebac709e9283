"""GPU: every specialised DP-fill kernel instantiation against the oracle.

One target automaton per (KC, KG, DEG, MV) tuple that dtw.cu compiles (tests/_layouts.py), each in a
noisy and a quantised form (levels and samples on a 1/8 grid, so candidates really tie).  For each
tuple: the automaton runs on the planned kernel; first-pass traces and end costs equal the oracle's
bit for bit; so do they for reads whose lengths put the band's first row and the last direction
word on every phase; masked second passes, with the end band closed and open, equal the oracle's;
the catch-all kernel gives the same traces and costs; and for regex loci the whole device call equals
the oracle's read by read."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import _layouts as lay
from oracle import caller_oracle as co
from warpstr_b200.config import CallerConfig

pytestmark = pytest.mark.gpu

CASES = lay.INSTANTIATIONS
THREADS = min(16, os.cpu_count() or 1)
N_NOISY, N_QUANT = 6, 4
CH = 126             # samples per signal tile of the fill kernel (WSTR_SIG_CHUNK)


class _Case:
    """A tuple's automata on the device and its reads (built once per module)."""

    def __init__(self, engine, case):
        from warpstr_b200 import _lib
        self.case, self.t, self.eng = case, lay.get(case), engine
        self.mv = case[3]
        self.noisy, self.quant = self.t.automaton(), self.t.automaton(quantised=True)
        self.id = {}
        for q, a in ((False, self.noisy), (True, self.quant)):
            self.id[('spec', q)] = engine.add_automaton(a, self.t.flank)
            self.id[('open', q)] = engine.add_automaton(a, self.t.flank_open)
        _lib.set_generic_only(True)
        try:
            for q, a in ((False, self.noisy), (True, self.quant)):
                self.id[('any', q)] = engine.add_automaton(a, self.t.flank)
        finally:
            _lib.set_generic_only(False)
        self.reads = [(x, False) for x in self.t.reads(N_NOISY, seed=11)] + \
                     [(x, True) for x in self.t.reads(N_QUANT, seed=12, quantised=True)]

        self.tb = {False: self.noisy.tables(), True: self.quant.tables()}

    def tables(self, quantised):
        return self.tb[quantised]

    def masks(self, flank, seed):
        return [band_mask(len(x), self.mv, flank, np.random.default_rng([seed, n])) for n, (x, _) in enumerate(self.reads)]


def band_mask(T, mv, flank, rng):
    """Masked rows (dwell mv-1) across 32-bit mask words, isolated rows, the rows below 2 mv, the end
    band's first rows and the read's last rows."""
    m = np.zeros(T, dtype=bool)
    for w in rng.integers(2, T // 32 - 1, 4):         # short stretches across a word boundary
        a = 32 * int(w) - int(rng.integers(1, 12))
        m[a:a + int(rng.integers(3, 24))] = True
    a = int(rng.integers(2 * mv, T - 200))
    m[a:a + 100] = True                                  # several whole words
    m[rng.integers(0, T, 30)] = True                     # isolated rows
    m[:2 * mv] = True
    band = max(6 * (flank - 10), T - 6 * (flank - 10) + 1)
    if band < T:
        m[max(0, band - 17):band + 23] = True
    m[T - 37:] = True
    return m


@pytest.fixture(scope='module')
def setup(built_lib):
    from warpstr_b200.caller import CallerEngine
    engines, cases = {}, {}

    def get(case):
        if case not in cases:
            mv = case[3]
            if mv not in engines:
                engines[mv] = CallerEngine(CallerConfig(min_values_per_state=mv))
            cases[case] = _Case(engines[mv], case)
        return cases[case]
    return get


def _oracle_traces(xs, tbs, masks, mv, flank):
    """cdp.warp of every read (reads of one automaton go through one warp_batch)."""
    from oracle import cdp
    out = [None] * len(xs)
    groups = {}
    for n, tb in enumerate(tbs):
        groups.setdefault(id(tb), (tb, []))[1].append(n)
    for tb, idx in groups.values():
        ms = [masks[n] if masks is not None else np.zeros(len(xs[n]), dtype=bool) for n in idx]
        got, _ = cdp.warp_batch([xs[n] for n in idx], tb, ms, mv, flank, threads=THREADS)
        for n, t in zip(idx, got):
            out[n] = t
    return out


def _oracle_fills(xs, tbs, mv, flank):
    from oracle import cdp
    with ThreadPoolExecutor(THREADS) as ex:
        return list(ex.map(lambda a: cdp.fill(a[0], a[1], np.zeros(len(a[0]), dtype=bool), mv, flank), zip(xs, tbs)))


def count_ties(x, tb, D, mv):
    """Cells of an unmasked fill whose winning candidate equals another candidate (stay, then the incoming
    edges), recomputed from the oracle's matrix.  Exact for quantised reads: every sum is exact there."""
    T = len(x)
    rows = np.arange(mv, T)
    ae = np.abs(x[:, None] - tb.values[None, :])
    C = np.cumsum(ae, axis=0)
    W = C[rows - 1] - C[rows - mv]                       # |x_t - v_p| for t = i-mv+1 .. i-1
    far = D[rows - mv] + W
    deg = np.diff(tb.in_ptr)
    cands = [D[rows - 1] + ae[rows]]
    for r in range(int(deg.max())):
        c = np.full_like(cands[0], np.inf)
        js = np.flatnonzero(deg > r)
        c[:, js] = far[:, tb.in_idx[tb.in_ptr[js] + r]] + ae[rows][:, js]
        cands.append(c)
    allc = np.stack(cands)
    best = allc.min(axis=0)
    tie = ((allc == best).sum(axis=0) >= 2) & np.isfinite(best) & (D[rows] == best)
    return int(tie.sum())


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_runs_on_the_planned_kernel(setup, case):
    c = setup(case)
    kc, kg, deg, mv = case
    for q in (False, True):
        info = c.eng.automata[c.id[('spec', q)]].info()
        assert (info['chain_slots'], info['generic_slots'], info['unrolled_in_degree']) == (kc, kg, deg)
        assert info['states_per_lane'] == kc + kg
        assert info['dir_bits_per_row'] == lay.dir_bits(kc, kg, deg)
        assert info['band_closed'] == 1
        a = c.eng.automata[c.id[('any', q)]].info()
        assert a['states_per_lane'] == 0 and a['unrolled_in_degree'] == 0
        assert c.eng.automata[c.id[('open', q)]].info()['band_closed'] == 0


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_first_pass(setup, case):
    c = setup(case)
    xs = [x for x, _ in c.reads]
    tbs = [c.tables(q) for _, q in c.reads]
    traces, costs = c.eng.warp_batch(xs, [c.id[('spec', q)] for _, q in c.reads], return_end_cost=True)
    want = _oracle_traces(xs, tbs, None, c.mv, c.t.flank)
    D = _oracle_fills(xs, tbs, c.mv, c.t.flank)
    ties = 0
    for n, (x, q) in enumerate(c.reads):
        assert np.array_equal(traces[n], want[n]), (case, n, np.flatnonzero(traces[n] != want[n])[:1])
        assert costs[n] == D[n][-1, tbs[n].endstate], (case, n)
        if q:
            ties += count_ties(x, tbs[n], D[n], c.mv)
    assert ties > 0, 'the quantised reads should make candidates tie'
    print(f'{lay.case_id(case)}: {ties} tied cells in {N_QUANT} quantised reads')


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_lengths_at_every_phase(setup, case):
    """One read cut to every length from T down to T - 2 RPW (mv-1): the band's first row and the last,
    partly filled direction word on every phase of both the word and the row cycle; lengths at both
    sides of a signal-tile boundary; the shortest reads the kernel takes."""
    c = setup(case)
    mv, rpw = c.mv, lay.rows_per_word(case)
    x, _ = c.reads[0]
    T = len(x)
    lengths = [T - k for k in range(2 * rpw * (mv - 1) + 1)]
    for m in (T // CH - 1, T // CH - 5):
        lengths += [CH * m + d for d in (-1, 0, 1, 2)]
    lengths += [mv + 1, mv + 2]
    xs = [np.ascontiguousarray(x[:n]) for n in lengths]
    aid = c.id[('spec', False)]
    traces, costs = c.eng.warp_batch(xs, [aid] * len(xs), return_end_cost=True)
    tb = c.tables(False)
    want = _oracle_traces(xs, [tb] * len(xs), None, mv, c.t.flank)
    D = _oracle_fills(xs, [tb] * len(xs), mv, c.t.flank)
    for n, L in enumerate(lengths):
        assert np.array_equal(traces[n], want[n]), (case, L)
        assert costs[n] == D[n][-1, tb.endstate], (case, L)
    with pytest.raises(IndexError):
        c.eng.warp_batch([np.ascontiguousarray(x[:mv])], [aid])


def _masked_pass(c, kind, flank, seed):
    xs = [x for x, _ in c.reads]
    tbs = [c.tables(q) for _, q in c.reads]
    masks = c.masks(flank, seed)
    got = c.eng.warp_batch(xs, [c.id[(kind, q)] for _, q in c.reads], masks)
    want = _oracle_traces(xs, tbs, masks, c.mv, flank)
    for n in range(len(xs)):
        assert np.array_equal(got[n], want[n]), (c.case, kind, n, np.flatnonzero(got[n] != want[n])[:1])


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_masked_pass(setup, case):
    c = setup(case)
    _masked_pass(c, 'spec', c.t.flank, seed=21)


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_open_end_band(setup, case):
    """A flank_length that puts the band's cut inside the ladder / repeat: back edges lead from kept
    states into skipped ones, so every banded row keeps the per-cell test.  Both passes."""
    c = setup(case)
    flank = c.t.flank_open
    xs = [x for x, _ in c.reads]
    tbs = [c.tables(q) for _, q in c.reads]
    traces, costs = c.eng.warp_batch(xs, [c.id[('open', q)] for _, q in c.reads], return_end_cost=True)
    want = _oracle_traces(xs, tbs, None, c.mv, flank)
    D = _oracle_fills(xs, tbs, c.mv, flank)
    for n in range(len(xs)):
        assert np.array_equal(traces[n], want[n]), (case, n, np.flatnonzero(traces[n] != want[n])[:1])
        assert costs[n] == D[n][-1, tbs[n].endstate], (case, n)
    _masked_pass(c, 'open', flank, seed=23)


@pytest.mark.parametrize('case', CASES, ids=lay.case_id)
def test_catch_all_gives_the_same(setup, case):
    """The same reads through the catch-all kernel: identical traces and end costs, both passes."""
    c = setup(case)
    xs = [x for x, _ in c.reads]
    masks = c.masks(c.t.flank, seed=21)
    got = []
    for kind in ('spec', 'any'):
        aut = [c.id[(kind, q)] for _, q in c.reads]
        t, e = c.eng.warp_batch(xs, aut, return_end_cost=True)
        got.append((t, e, c.eng.warp_batch(xs, aut, masks)))
    for n in range(len(xs)):
        assert np.array_equal(got[0][0][n], got[1][0][n]), (case, n)
        assert np.array_equal(got[0][2][n], got[1][2][n]), (case, n, 'masked')
    assert np.array_equal(got[0][1], got[1][1])


@pytest.mark.parametrize('case', sorted(lay.REGEX), ids=lay.case_id)
def test_whole_call(setup, case):
    """wstr_call_batch on the regex targets: both traces, the rescaled signal, sequences and costs bit
    for bit against the oracle's run of the read (the second pass runs on the mid-stage's own masks)."""
    c = setup(case)
    xs = [x for x, q in c.reads if not q]
    aut = [c.id[('spec', False)]] * len(xs)
    rev = [c.t.reverse] * len(xs)
    packed = c.eng.upload(xs, aut, rev)
    o = c.eng.call_packed(*packed, want_debug=True)
    off, lengths = packed[1], packed[2]
    assert not o['status'].cpu().numpy().any()
    t1, t2, resc = o['trace1'].cpu().numpy(), o['trace2'].cpu().numpy(), o['rescaled'].cpu().numpy()
    res = c.eng.results_from(o, xs, aut, rev)
    tb, kn = c.tables(False), co.Knobs(min_values_per_state=c.mv)
    with ThreadPoolExecutor(THREADS) as ex:
        wants = list(ex.map(lambda x: co.run_read(x, tb, c.t.flank, c.t.reverse, kn=kn, impl='c'), xs))
    for n, want in enumerate(wants):
        a, ln = int(off[n]), int(lengths[n])
        assert np.array_equal(t1[a:a + ln], want.trace1), (case, n)
        assert np.array_equal(resc[a:a + ln], want.rescaled), (case, n)
        assert np.array_equal(t2[a:a + ln], want.trace2), (case, n)
        assert res[n].seq == want.seq and res[n].resc_seq == want.resc_seq, (case, n)
        assert res[n].cost == want.cost and res[n].resc_cost == want.resc_cost, (case, n)


def test_every_instantiation_in_one_batch_and_waves(built_lib):
    """Every target of a dwell setting in one batch (a batch holds one dwell), first and masked pass, with a
    workspace so small that the batch runs in several waves."""
    from warpstr_b200 import _lib
    from warpstr_b200.caller import CallerEngine
    for mv in sorted({case[3] for case in CASES}):
        eng = CallerEngine(CallerConfig(min_values_per_state=mv))
        xs, aut, tbs, flanks, masks = [], [], [], [], []
        for case in (k for k in CASES if k[3] == mv):
            t = lay.get(case)
            for q in (False, True):
                aid = eng.add_automaton(t.automaton(q), t.flank)
                for n, x in enumerate(t.reads(2, seed=31, quantised=q)):
                    xs.append(x); aut.append(aid); tbs.append(t.automaton(q).tables()); flanks.append(t.flank)
                    masks.append(band_mask(len(x), mv, t.flank, np.random.default_rng([mv, len(xs)])))
        need = _lib.warp_workspace_bytes(eng.automata, np.asarray(aut, dtype=np.int32),
                                         np.asarray([len(x) for x in xs], dtype=np.int32))
        eng.workspace_limit = max(need // 4, 1 << 20)
        assert need > 2 * eng.workspace_limit
        order = np.random.default_rng(mv).permutation(len(xs))     # automata interleaved in the batch
        xs = [xs[i] for i in order]; aut = [aut[i] for i in order]; tbs = [tbs[i] for i in order]
        flanks = [flanks[i] for i in order]; masks = [masks[i] for i in order]
        from oracle import cdp
        for ms in (None, masks):
            got = eng.warp_batch(xs, aut, ms)
            with ThreadPoolExecutor(THREADS) as ex:
                want = list(ex.map(lambda n: cdp.warp(xs[n], tbs[n], np.zeros(len(xs[n]), dtype=bool) if ms is None
                                                      else ms[n], mv, flanks[n]), range(len(xs))))
            for n in range(len(xs)):
                assert np.array_equal(got[n], want[n]), (mv, n, ms is not None)
