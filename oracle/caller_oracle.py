"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the WarpSTR per-read caller.

Restates, function by function, what /root/reference/src/caller/caller.py computes
for one read, over flat automaton tables (values, seq_idx, CSR incoming) instead of
State objects.  It exists to check the CUDA path and to serve as the timed CPU
baseline; the product never imports it.

Pinning: every function here is compared with the unmodified reference code (imported
through oracle/refshim.py in the build container) by tests/test_oracle_pinned.py, and
with the committed golden vectors in tests/golden/ (generated from the reference by
oracle/make_golden.py) wherever the reference tree is absent.  The reference itself
holds no unit-level vectors for this path (SURVEY.md section 4); its one end-to-end
figure (README.md:55) needs GRCh38 + VBZ fast5 and is not reachable here.

Three DP formulations, all float64 and all producing bit-identical matrices:
  fill_scalar   -- cell-by-cell loops in the reference's own order (slow, the timed
                   "port" of the reference's Python DP)
  fill_rows     -- one numpy vector operation per row and per incoming rank
  dp_oracle.c   -- the same loops in C (oracle/dp_oracle.c, via ctypes)
"""
from dataclasses import dataclass
from math import sqrt
from typing import List, Optional, Sequence

import numpy as np
from scipy import interpolate


@dataclass
class Tables:
    values: np.ndarray      # f64[S]
    seq_idx: np.ndarray     # i32[S]
    in_ptr: np.ndarray      # i32[S+1]
    in_idx: np.ndarray      # i32[E]
    rep_mask: np.ndarray    # bool[S]
    last_base: str          # S characters
    endstate: int

    @property
    def n_states(self):
        return len(self.values)


def tables_from(automaton) -> Tables:
    """Accepts the reference's StateAutomata or any object with .states/.mask/.endstate."""
    st = automaton.states
    ptr = np.zeros(len(st) + 1, dtype=np.int32)
    idx: List[int] = []
    for i, s in enumerate(st):
        idx.extend(p.idx for p in s.incoming)
        ptr[i + 1] = len(idx)
    return Tables(values=np.array([s.value for s in st], dtype=np.float64),
                  seq_idx=np.array([s.seq_idx for s in st], dtype=np.int32),
                  in_ptr=ptr, in_idx=np.array(idx, dtype=np.int32),
                  rep_mask=np.array(automaton.mask, dtype=bool),
                  last_base=''.join(s.kmer[-1] for s in st),
                  endstate=int(automaton.endstate))


@dataclass
class Knobs:
    """The configuration values the per-read path reads (src/default.yaml:7-23)."""
    min_values_per_state: int = 4
    states_in_segment: int = 6
    reps_as_one: bool = False
    threshold: float = 0.5
    max_std: float = 0.5
    method: str = 'mean'


# --------------------------------------------------------------------------------------
# DP fill (caller.py:198-245)
# --------------------------------------------------------------------------------------
def _band(tb: Tables, T: int, flank_length: int):
    # caller.py:211-214
    boundary = flank_length - 10
    after_repeat = int(tb.seq_idx[-1]) - boundary
    return 6 * boundary, T - 6 * boundary, after_repeat


def fill_scalar(x: np.ndarray, tb: Tables, mask: np.ndarray, mv: int, flank_length: int) -> np.ndarray:
    """Cell-by-cell float64 DP exactly as the reference iterates it (caller.py:198-245)."""
    T, S = len(x), tb.n_states
    inf = float('inf')
    D = np.full((T, S), np.inf)
    v = [float(a) for a in tb.values]
    sig = [float(a) for a in x]
    sq = [int(a) for a in tb.seq_idx]
    inc = [[int(p) for p in tb.in_idx[tb.in_ptr[j]:tb.in_ptr[j + 1]]] for j in range(S)]
    first = abs(sig[0] - v[0])
    D[0, 0] = first
    for c in range(1, mv + 1):                       # row 0, *column* c (caller.py:206-208)
        D[0, c] = first + abs(sig[c] - v[0])
    th1, th2, after = _band(tb, T, flank_length)
    for i in range(mv, T):
        back = mv - 1 if mask[i] else mv
        xi = sig[i]
        row, prev_row, far_row = D[i], D[i - 1], D[i - back]
        for j in range(S):
            if i < th1:
                if i < sq[j] * 4 and i > sq[j] * 15:   # never true (caller.py:220-222)
                    continue
            elif i > th2 and sq[j] < after:
                continue
            emit = abs(xi - v[j])
            best = inf
            up = prev_row[j]
            if up != inf:
                c = up + emit
                if c < best:
                    best = c
            for p in inc[j]:
                c = far_row[p]
                if c == inf:
                    continue
                vp = v[p]
                for t in range(i - back + 1, i):
                    c += abs(sig[t] - vp)
                c += emit
                if c < best:
                    best = c
            row[j] = best
    return D


def fill_rows(x: np.ndarray, tb: Tables, mask: np.ndarray, mv: int, flank_length: int):
    """Row-vectorised DP.  Returns (D, ptr) where ptr[i, j] = 0 for 'stay', r+1 for
    incoming[r]; same additions in the same order as fill_scalar, so D is bit-identical."""
    T, S = len(x), tb.n_states
    v = tb.values
    D = np.full((T, S), np.inf)
    ptr = np.zeros((T, S), dtype=np.int8)
    first = abs(x[0] - v[0])
    D[0, 0] = first
    for c in range(1, mv + 1):
        D[0, c] = first + abs(x[c] - v[0])
    deg = np.diff(tb.in_ptr)
    maxdeg = int(deg.max()) if S else 0
    pred = np.full((maxdeg, S), -1, dtype=np.int64)
    for j in range(S):
        lst = tb.in_idx[tb.in_ptr[j]:tb.in_ptr[j + 1]]
        pred[:len(lst), j] = lst
    has = pred >= 0
    predc = np.where(has, pred, 0)
    th1, th2, after = _band(tb, T, flank_length)
    skip_cols = tb.seq_idx < after
    E = np.abs(x[:, None] - v[None, :]) if T * S <= 4_000_000 else None
    for i in range(mv, T):
        back = mv - 1 if mask[i] else mv
        emit = E[i] if E is not None else np.abs(x[i] - v)
        best = np.full(S, np.inf)
        code = np.zeros(S, dtype=np.int8)
        c = D[i - 1] + emit
        take = c < best
        best = np.where(take, c, best)
        for r in range(maxdeg):
            p = predc[r]
            c = D[i - back][p]
            for t in range(i - back + 1, i):
                et = E[t] if E is not None else np.abs(x[t] - v)
                c = c + et[p]
            c = c + emit
            take = has[r] & (c < best)
            best = np.where(take, c, best)
            code = np.where(take, r + 1, code)
        if i >= th1 and i > th2:
            best = np.where(skip_cols, np.inf, best)
            code = np.where(skip_cols, 0, code)
        D[i] = best
        ptr[i] = code
    return D, ptr


# --------------------------------------------------------------------------------------
# traceback (caller.py:247-301)
# --------------------------------------------------------------------------------------
def backtrack_closest(D: np.ndarray, x: np.ndarray, tb: Tables, mask: np.ndarray, mv: int) -> np.ndarray:
    """The reference's traceback: recompute every candidate of the current cell and
    follow the one closest to the stored value; a skip must be strictly closer than
    'stay', the first incoming state wins ties."""
    v = tb.values
    j = tb.endstate
    i = len(D) - 1
    out: List[int] = []
    chosen = -1
    while i != 0:
        here = D[i][j]
        if D[i - 1][j] == np.inf:
            d_stay = np.inf
        else:
            d_stay = abs((D[i - 1][j] + abs(x[i] - v[j])) - here)
        back = mv - 1 if mask[i] else mv
        d_skip = np.inf
        for p in tb.in_idx[tb.in_ptr[j]:tb.in_ptr[j + 1]]:
            c = D[i - back][p]
            if c == np.inf:
                continue
            for t in range(i - back + 1, i):
                c += abs(x[t] - v[p])
            c += abs(x[i] - v[j])
            d = abs(c - here)
            if d < d_skip:
                d_skip, chosen = d, int(p)
        out.append(j)
        if d_skip < d_stay:
            if chosen == -1:
                raise RuntimeError('Unexpected error during backtracking')
            out.extend([chosen] * (back - 1))
            i -= back
            j = chosen
        else:
            i -= 1
    out.append(j)
    return np.asarray(out, dtype=int)[::-1]


def backtrack_ptr(ptr: np.ndarray, tb: Tables, mask: np.ndarray, mv: int) -> np.ndarray:
    """Traceback that follows stored arg-min codes (what the GPU does)."""
    j = tb.endstate
    i = ptr.shape[0] - 1
    out: List[int] = []
    while i != 0:
        code = int(ptr[i, j])
        out.append(j)
        if code == 0:
            i -= 1
        else:
            back = mv - 1 if mask[i] else mv
            p = int(tb.in_idx[tb.in_ptr[j] + code - 1])
            out.extend([p] * (back - 1))
            i -= back
            j = p
    out.append(j)
    return np.asarray(out, dtype=int)[::-1]


def warp(x: np.ndarray, tb: Tables, mask: Optional[Sequence[bool]], kn: Knobs, flank_length: int,
         impl: str = 'rows') -> np.ndarray:
    """caller.py:189-193.  An empty / None mask means 'no masked rows'."""
    m = np.asarray(mask, dtype=bool) if mask is not None and len(mask) else np.full(len(x), False)
    if impl == 'scalar':
        D = fill_scalar(x, tb, m, kn.min_values_per_state, flank_length)
        return backtrack_closest(D, x, tb, m, kn.min_values_per_state)
    if impl == 'c':
        from . import cdp
        return cdp.warp(x, tb, m, kn.min_values_per_state, flank_length)
    D, ptr = fill_rows(x, tb, m, kn.min_values_per_state, flank_length)
    return backtrack_ptr(ptr, tb, m, kn.min_values_per_state)


# --------------------------------------------------------------------------------------
# between the two passes (caller.py:58-96, 304-421)
# --------------------------------------------------------------------------------------
def state_transitions(trace: np.ndarray) -> np.ndarray:
    # caller.py:58-60
    keep = np.insert(np.diff(trace).astype(bool), 0, True)
    return trace[keep]


@dataclass
class RunStat:
    raw_values: list
    expected: float
    state_value: float


def _collapse(kn: Knobs, vals):
    if kn.method == 'mean':
        return np.average(vals)
    if kn.method == 'median':
        return np.median(vals)
    raise KeyError(f'Invalid alignment method: {kn.method}')


def create_alignment(trace: np.ndarray, x: np.ndarray, tb: Tables, kn: Knobs) -> List[RunStat]:
    # caller.py:65-96
    out: List[RunStat] = []
    trans = state_transitions(trace)
    if kn.reps_as_one:
        for s in np.unique(trans):
            raws = np.take(x, np.where(trace == s)[0])
            out.append(RunStat(raws, tb.values[s], _collapse(kn, raws)))
        return out
    pos = 0
    T = len(trace)
    for s in trans:
        raws = []
        while pos < T and trace[pos] == s:
            raws.append(x[pos])
            pos += 1
        out.append(RunStat(raws, tb.values[s], _collapse(kn, raws)))
    return out


def good_enough(r: RunStat, kn: Knobs) -> bool:
    # caller.py:23-39
    return bool(len(r.raw_values) >= kn.min_values_per_state
                and np.std(r.raw_values) < kn.max_std
                and abs(r.expected - r.state_value) <= kn.threshold)


def rescale_signal(x: np.ndarray, runs: List[RunStat], kn: Knobs) -> np.ndarray:
    # caller.py:304-318
    pairs = [(r.state_value, r.expected) for r in runs if good_enough(r, kn)]
    pairs.sort(key=lambda t: t[0])
    xs = [p[0] for p in pairs]
    ys = [p[1] for p in pairs]
    tck = interpolate.splrep(xs, ys, s=len(xs))
    return interpolate.splev(x, tck)


def _ttest(a: np.ndarray, b: np.ndarray, win: int) -> float:
    # caller.py:347-354
    sd = sqrt((np.std(a) ** 2 + np.std(b) ** 2) / win)
    if sd == 0:
        sd = sd + 0.0000001
    return (np.mean(a) - np.mean(b)) / sd


def segment_count(data: np.ndarray, win: int) -> int:
    # caller.py:357-378
    stats = [_ttest(data[c - win:c], data[c:c + win], win) for c in range(win, len(data) - win + 1)]
    borders = []
    rising = False
    prev = stats[0]
    for n, t in enumerate(stats):
        if t > 3 or t < -3:
            if (t > 3 and t >= prev) or (t < -3 and t <= prev):
                rising = True
            else:
                if rising:
                    borders.append(n + win - 1)
                rising = False
        elif rising:
            borders.append(n + win - 1)
            rising = False
        prev = t
    return len(borders) - 1


def find_event_borders(rep_mask, trace: np.ndarray, trans: np.ndarray, kn: Knobs):
    # caller.py:381-406
    sis = kn.states_in_segment
    in_rep = [n for n, s in enumerate(trans) if rep_mask[s]]
    start, end = in_rep[0], in_rep[-1]

    def span(a, b):
        lo = np.where(trace == trans[a])[0][0]
        hi = np.where(trace == trans[b])[0][-1]
        cuts = np.where(np.diff(trace[lo:hi + 1]).astype(bool))[0]
        return lo, hi, cuts

    lo, hi, cuts = span(start, end)
    extra = (len(cuts) - 1) % sis
    if extra > 0:
        end = end + (sis - extra)
        lo, hi, cuts = span(start, end)
    cuts = lo + cuts
    bounds = [c for n, c in enumerate(cuts) if n % sis == 0]
    return start, end, lo, hi, bounds


def mask_bad_repeats(x: np.ndarray, rep_mask, trace: np.ndarray, trans: np.ndarray, kn: Knobs):
    # caller.py:330-344, 409-421
    start, end, lo, hi, bounds = find_event_borders(rep_mask, trace, trans, kn)
    win = 3
    counts = [segment_count(x[bounds[n] - win:b + win], win) for n, b in enumerate(bounds[1:])]
    bad = [n for n, c in enumerate(counts) if c >= kn.states_in_segment + 1]
    out = [False] * lo
    out += [False] * (bounds[0] - lo)
    for n in range(len(bounds) - 1):
        out += [n in bad] * (bounds[n + 1] - bounds[n])
    out += [False] * (hi - bounds[-1])
    out += [False] * (len(x) - hi)
    return start, end, out


# --------------------------------------------------------------------------------------
# bulk variants: the same arithmetic on array slices / whole windows instead of Python lists
# per sample, ~3x faster per read; pinned against the functions above (and so against the
# reference) by tests/test_oracle_golden.py::test_bulk_oracle_equals_the_plain_one
# --------------------------------------------------------------------------------------
def create_alignment_bulk(trace: np.ndarray, x: np.ndarray, tb: Tables, kn: Knobs) -> List[RunStat]:
    if kn.reps_as_one:
        return create_alignment(trace, x, tb, kn)
    cut = np.flatnonzero(trace[1:] != trace[:-1]) + 1
    starts = np.concatenate(([0], cut))
    ends = np.concatenate((cut, [len(trace)]))
    return [RunStat(x[a:b], tb.values[trace[a]], _collapse(kn, x[a:b])) for a, b in zip(starts, ends)]


def _tstat_terms(data: np.ndarray, win: int):
    """Numerator and denominator of the t statistic at every centre of `data` (caller.py:347-354, 358),
    the denominator before a zero is replaced: np.mean / np.std of 3 samples are sequential sums; the
    squares are libm pow(x, 2.0) -- what `np.float64 ** 2` evaluates to."""
    from math import pow as libm_pow
    assert win == 3
    n = len(data) - 2 * win + 1
    if n <= 0:
        return np.zeros(0), np.zeros(0)
    w = np.lib.stride_tricks.sliding_window_view(data, win)          # w[c] = data[c:c+3]

    mean = ((w[:, 0] + w[:, 1]) + w[:, 2]) / 3
    d = w - mean[:, None]
    sd = np.sqrt(((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) / 3)
    sq = np.fromiter((libm_pow(v, 2.0) for v in sd.tolist()), dtype=np.float64, count=len(sd))
    den = np.sqrt((sq[:n] + sq[win:win + n]) / win)
    return mean[:n] - mean[win:win + n], den


def _tstats_bulk(data: np.ndarray, win: int) -> List[float]:
    num, den = _tstat_terms(data, win)
    den = np.where(den == 0, den + 0.0000001, den)
    return (num / den).tolist()


def zero_sd_windows(x: np.ndarray, rep_mask, trace: np.ndarray, kn: Knobs) -> int:
    """How many t statistics of the bad-repeat mask of ``x`` along ``trace`` have two windows of zero
    deviation, i.e. divide by the 1e-7 of caller.py:352-353 (for reads the mask does not raise on)."""
    _, _, _, _, bounds = find_event_borders(rep_mask, trace, state_transitions(trace), kn)
    return sum(int((_tstat_terms(x[bounds[n] - 3:b + 3], 3)[1] == 0).sum()) for n, b in enumerate(bounds[1:]))


def segment_count_bulk(data: np.ndarray, win: int) -> int:
    stats = _tstats_bulk(data, win)
    n_borders = 0
    rising = False
    prev = stats[0]                       # IndexError on an empty window, like the reference
    for t in stats:
        if t > 3 or t < -3:
            if (t > 3 and t >= prev) or (t < -3 and t <= prev):
                rising = True
            else:
                if rising:
                    n_borders += 1
                rising = False
        elif rising:
            n_borders += 1
            rising = False
        prev = t
    return n_borders - 1


def mask_bad_repeats_bulk(x: np.ndarray, rep_mask, trace: np.ndarray, trans: np.ndarray, kn: Knobs):
    start, end, lo, hi, bounds = find_event_borders(rep_mask, trace, trans, kn)
    win = 3
    counts = [segment_count_bulk(x[bounds[n] - win:b + win], win) for n, b in enumerate(bounds[1:])]
    out = np.zeros(len(x), dtype=bool)
    for n, c in enumerate(counts):
        if c >= kn.states_in_segment + 1:
            out[bounds[n]:bounds[n + 1]] = True
    _ = bounds[0]
    return start, end, out


# --------------------------------------------------------------------------------------
# whole read (caller.py:117-149, 178-187)
# --------------------------------------------------------------------------------------
_COMP = str.maketrans('ACGTN', 'TGCAN')


def decode_sequence(trace: np.ndarray, tb: Tables, flank_length: int, reverse: bool) -> str:
    trans = state_transitions(trace)
    seq = ''.join(tb.last_base[s] for s in trans)
    offset = int(tb.seq_idx[trans[0]])
    seq = seq[flank_length - offset:-flank_length]
    return seq.translate(_COMP)[::-1] if reverse else seq


@dataclass
class OracleResult:
    seq: str
    cost: float
    resc_seq: str
    resc_cost: float
    trace1: np.ndarray
    trace2: np.ndarray
    rescaled: np.ndarray
    badmask: np.ndarray


@dataclass
class FirstPass:
    """What the reference derives from the first pass's trace (caller.py:123-126, 138)."""
    alignment: List[RunStat]
    rescaled: np.ndarray
    badmask: np.ndarray
    start: int
    end: int
    cost: float


@dataclass
class SecondPass:
    """What the reference derives from the second pass's trace (caller.py:132-135, 139)."""
    start: int
    end: int
    cost: float


def _state_cost(runs: List[RunStat], start: int, end: int) -> float:
    # caller.py:138-139
    return np.mean([abs(r.state_value - r.expected) for r in runs[start:end]])


def after_first_pass(x: np.ndarray, t1: np.ndarray, tb: Tables, kn: Knobs, bulk: bool = False) -> FirstPass:
    """The mid-stage between the passes: alignment of ``x`` along ``t1``, rescaled signal, bad-repeat mask,
    repeat region and state-wise cost.  Raises what the reference raises for the read."""
    align = create_alignment_bulk if bulk else create_alignment
    mask_of = mask_bad_repeats_bulk if bulk else mask_bad_repeats
    runs = align(t1, x, tb, kn)
    resc = rescale_signal(x, runs, kn)
    start, end, bad = mask_of(x, tb.rep_mask, t1, state_transitions(t1), kn)
    return FirstPass(alignment=runs, rescaled=np.asarray(resc), badmask=np.asarray(bad, dtype=bool),
                     start=start, end=end, cost=_state_cost(runs, start, end))


def after_second_pass(resc: np.ndarray, t2: np.ndarray, tb: Tables, kn: Knobs, bulk: bool = False) -> SecondPass:
    """The stage after the second pass: the rescaled signal is rescaled again only to find the repeat region
    (its mask is not used); returns that region and the state-wise cost."""
    align = create_alignment_bulk if bulk else create_alignment
    mask_of = mask_bad_repeats_bulk if bulk else mask_bad_repeats
    runs = align(t2, resc, tb, kn)
    resc2 = rescale_signal(resc, runs, kn)
    start, end, _ = mask_of(resc2, tb.rep_mask, t2, state_transitions(t2), kn)
    return SecondPass(start=start, end=end, cost=_state_cost(runs, start, end))


def run_read(x: np.ndarray, tb: Tables, flank_length: int, reverse: bool,
             kn: Optional[Knobs] = None, impl: str = 'rows', bulk: bool = False) -> OracleResult:
    """``bulk``: the array-slice variants of the mid-stage (same arithmetic, ~3x faster)."""
    kn = kn or Knobs()
    x = np.asarray(x, dtype=np.float64)
    t1 = warp(x, tb, None, kn, flank_length, impl)
    p1 = after_first_pass(x, t1, tb, kn, bulk)
    t2 = warp(p1.rescaled, tb, p1.badmask, kn, flank_length, impl)
    p2 = after_second_pass(p1.rescaled, t2, tb, kn, bulk)
    return OracleResult(seq=decode_sequence(t1, tb, flank_length, reverse), cost=p1.cost,
                        resc_seq=decode_sequence(t2, tb, flank_length, reverse), resc_cost=p2.cost,
                        trace1=t1, trace2=t2, rescaled=p1.rescaled, badmask=p1.badmask)
