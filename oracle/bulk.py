"""TEST INFRASTRUCTURE ONLY -- the oracle over thousands of reads, spread over a process pool on the host
cores.  ``run_reads``: the whole ``run_read(impl='c', bulk=True)`` (the DP in C, the mid-stage on array
slices), used by the bulk parity tests and by bench.py's `parity` object.  ``run_midstage``: the mid-stage
alone on traces the device produced, with facts about which branches of the device's mid-stage the read
takes.  Never used by the product."""
import multiprocessing as mp
import os
from typing import List, Sequence, Tuple

import numpy as np

_CTX = {}


def _init(regexes: Sequence[str], flank_length: int, knobs):
    from oracle import caller_oracle as co
    from oracle import cdp
    from warpstr_b200.automata import StateAutomata
    cdp.build()
    _CTX['co'] = co
    _CTX['tb'] = [co.tables_from(StateAutomata(rx)) for rx in regexes]
    _CTX['F'] = flank_length
    _CTX['kn'] = co.Knobs(*knobs) if knobs is not None else None


def _one(job) -> Tuple:
    sig, aut, rev, want_traces = job
    co = _CTX['co']
    try:
        r = co.run_read(sig, _CTX['tb'][aut], _CTX['F'], bool(rev), _CTX['kn'], impl='c', bulk=True)
    except Exception as exc:                       # what the reference would raise for this read
        return ('error', type(exc).__name__)
    out = (r.seq, r.resc_seq, float(r.cost), float(r.resc_cost))
    if want_traces:
        out += (r.trace1.astype(np.int32), r.trace2.astype(np.int32))
    return out


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _pool_map(fn, jobs, regexes, flank_length, knobs, workers):
    workers = workers or host_cores()
    if workers <= 1 or len(jobs) < 4:
        _init(regexes, flank_length, knobs)
        return [fn(j) for j in jobs]
    with mp.get_context('fork').Pool(workers, initializer=_init, initargs=(list(regexes), flank_length, knobs)) as pool:
        return pool.map(fn, jobs, chunksize=max(1, len(jobs) // (workers * 8)))


def run_reads(regexes: Sequence[str], flank_length: int, signals: Sequence[np.ndarray], aut: Sequence[int],
              rev: Sequence[bool], knobs=None, want_traces: bool = False, workers: int = 0) -> List[Tuple]:
    """Oracle results, in order: (seq, resc_seq, cost, resc_cost[, trace1, trace2]) or ('error', type name).
    ``regexes[a]`` is the automaton regex of automaton id ``a``; ``knobs`` the Knobs fields as a tuple."""
    jobs = [(np.ascontiguousarray(s, dtype=np.float64), int(a), bool(r), want_traces)
            for s, a, r in zip(signals, aut, rev)]
    return _pool_map(_one, jobs, regexes, flank_length, knobs, workers)


def _error_status(exc: Exception, trace: np.ndarray, tb) -> int:
    """The device's WSTR_READ_* code for what the reference raises in the mid-stage (include/warpstr_b200.h)."""
    if isinstance(exc, IndexError):
        return 6 if tb.rep_mask[np.unique(trace)].any() else 3    # trues[0] of a path without a repeat state
    if isinstance(exc, (TypeError, ValueError)):                  # splrep's input checks
        return 4
    return -1


def _mid_one(job) -> dict:
    x, t1, t2, aut, rev = job
    co, tb, kn, F = _CTX['co'], _CTX['tb'][aut], _CTX['kn'] or _CTX['co'].Knobs(), _CTX['F']
    out = {'status': 0, 'error': None}
    try:
        p1 = co.after_first_pass(x, t1, tb, kn, bulk=True)
    except Exception as exc:
        return dict(out, status=_error_status(exc, t1, tb), error=type(exc).__name__)
    good = [r for r in p1.alignment if co.good_enough(r, kn)]
    keys = np.array([r.state_value for r in good])
    _, counts = np.unique(keys, return_counts=True)
    cut = np.flatnonzero(t1[1:] != t1[:-1]) + 1
    runs = np.diff(np.concatenate(([0], cut, [len(t1)])))
    out.update(rescaled=p1.rescaled, mask=p1.badmask, cost1=float(p1.cost), seq1=co.decode_sequence(t1, tb, F, rev),
               m=len(good), ties=int(counts[counts > 1].sum()), run_hist=np.bincount(runs),
               groups=np.array([len(r.raw_values) for r in p1.alignment]) if kn.reps_as_one else np.zeros(0, int),
               zero_sd=co.zero_sd_windows(x, tb.rep_mask, t1, kn))
    try:
        p2 = co.after_second_pass(p1.rescaled, t2, tb, kn, bulk=True)
    except Exception as exc:
        return dict(out, status=_error_status(exc, t2, tb), error=type(exc).__name__)
    out.update(cost2=float(p2.cost), seq2=co.decode_sequence(t2, tb, F, rev))
    return out


def run_midstage(regexes: Sequence[str], flank_length: int, signals: Sequence[np.ndarray],
                 traces1: Sequence[np.ndarray], traces2: Sequence[np.ndarray], aut: Sequence[int],
                 rev: Sequence[bool], knobs=None, workers: int = 0) -> List[dict]:
    """The oracle's mid-stage applied to each read's signal and the two traces the device took for it (no DP
    on the host).  Per read a dict: ``status`` (0, or the WSTR_READ_* code of what the reference raises, with
    ``error`` its type name), and, as far as the read got, ``rescaled``, ``mask``, ``cost1``, ``seq1``,
    ``cost2``, ``seq2`` and the coverage facts of the first pass: ``run_hist`` (bincount of the run lengths of
    trace1), ``m`` (good pairs), ``ties`` (good pairs whose key another good pair shares), ``groups`` (sizes of
    the alignment entries under reps_as_one) and ``zero_sd`` (see ``zero_sd_windows``)."""
    jobs = [(np.ascontiguousarray(s, dtype=np.float64), np.asarray(t1), np.asarray(t2), int(a), bool(r))
            for s, t1, t2, a, r in zip(signals, traces1, traces2, aut, rev)]
    return _pool_map(_mid_one, jobs, regexes, flank_length, knobs, workers)
