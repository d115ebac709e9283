"""The caller seam: ``CallerWrapper(locus, threads).run(workload) -> List[CallerResult]``.

Drop-in for the reference's ``CallerWrapper`` (caller/wrapper.py:57-248): builds the
template- and reverse-strand automata from the locus regex and its flanks, runs every read
of the workload (order preserved) and offers the same helpers for complex loci
(``break_into_units``, ``collapse_repeats``).  Where the reference fans reads out to a
``multiprocessing.Pool`` (:104-120), this sends the whole workload to the GPU in one batch;
``threads`` is accepted for signature compatibility and ignored.
"""
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import pandas as pd

from . import templates as tmpl
from .automata import StateAutomata
from .caller import CallerEngine, CallerResult, _VBZReads, _WholeReads, fill_given_strands, pack_raw, pack_vbz
from .config import CallerConfig, Config, RescalerConfig
from .pore_model import PoreModel, get_pore_model


@dataclass
class ReadSignal:
    """schemas/readsignal.py:6-10"""
    name: str
    reverse: bool
    signal: np.ndarray


@dataclass
class Flank:
    left: str
    right: str


@dataclass
class Flanks:
    template: Flank
    reverse: Flank


def load_flanks(path: str) -> Flanks:
    """Flanks written by the expected-signal step (``expected_signals/sequences.csv``,
    lines ``type,sequence``; reference: extractor/tr_extractor.py:108-140)."""
    fname = os.path.join(path, tmpl.LOCUS_INFO_SUBDIR, tmpl.LOCUS_FLANKS)
    seqs = {}
    with open(fname, 'r') as fh:
        next(fh)
        for line in fh:
            parts = line.strip().split(',')
            if len(parts) == 2:
                seqs[parts[0]] = parts[1]
    try:
        return Flanks(template=Flank(seqs['left_flank_template'], seqs['right_flank_template']),
                      reverse=Flank(seqs['left_flank_reverse'], seqs['right_flank_reverse']))
    except KeyError as exc:
        raise KeyError(f'{fname} lacks the flank {exc}')


def flanks_from_template(left: str, right: str) -> Flanks:
    """Reverse-strand flanks are the swapped reverse complements (dna_sequence.py:54-55)."""
    return Flanks(template=Flank(left, right),
                  reverse=Flank(tmpl.reverse_complement(right), tmpl.reverse_complement(left)))


@dataclass
class Locus:
    """The fields of the reference's Locus that the caller reads (schemas/locus.py:8-46).
    ``sequence`` must be given; deriving it from ``motif`` needs the reference genome and is
    outside this path."""
    name: str
    sequence: str
    flank_length: int = 110
    path: str = ''
    coord: str = ''

    def __post_init__(self):
        self.sequence = self.sequence.upper()


class CallerWrapper:
    def __init__(self, locus: Locus, threads: int = 1, flanks: Optional[Flanks] = None,
                 caller_config: Optional[CallerConfig] = None, rescaler_config: Optional[RescalerConfig] = None,
                 pore_model: Optional[PoreModel] = None, engine: Optional[CallerEngine] = None,
                 config: Optional[Config] = None):
        if config is not None:
            caller_config = caller_config or config.caller_config
            rescaler_config = rescaler_config or config.rescaler_config
        self.locus = locus
        self.threads = threads
        self.caller_config = caller_config or CallerConfig()
        self.pore_model = pore_model or get_pore_model()
        self.flanks = flanks if flanks is not None else load_flanks(locus.path)
        template_seq, reverse_seq = self.get_seqs(locus.sequence, self.flanks)
        if locus.path and os.path.isdir(os.path.join(locus.path, tmpl.SUMMARY_SUBDIR)):
            self.check_high_similarity(locus.sequence)
        self.units, self.repeat_units, self.offsets = self.break_into_units(locus.sequence)
        self.temp_sta = StateAutomata(template_seq, self.pore_model)
        self.rev_sta = StateAutomata(reverse_seq, self.pore_model)
        self.engine = engine or CallerEngine(self.caller_config, rescaler_config)
        self._temp_id = self.engine.add_automaton(self.temp_sta, locus.flank_length)
        self._rev_id = self.engine.add_automaton(self.rev_sta, locus.flank_length)

    # -- sequences (wrapper.py:72-84) --------------------------------------------------------------
    def get_seqs(self, sequence: str, flanks: Flanks):
        tmp = flanks.template.left + sequence + flanks.template.right
        rev = flanks.reverse.left + self.reverse_uniq_sequence(sequence) + flanks.reverse.right
        return tmp, rev

    @staticmethod
    def reverse_uniq_sequence(sequence: str) -> str:
        return tmpl.reverse_uniq_sequence(sequence)

    # -- the call (wrapper.py:104-120) ---------------------------------------------------------------
    def run(self, workload: Sequence[ReadSignal]) -> List[CallerResult]:
        """The reference's call: float64 STR windows, each with its strand (a None strand raises ValueError)."""
        signals = [np.ascontiguousarray(r.signal, dtype=np.float64) for r in workload]
        reverse = _strands([r.reverse for r in workload])
        _need_strands(reverse, [r.name for r in workload], 'a ReadSignal')
        aut = self._aut(reverse)
        return self.engine.call_batch(signals, aut, reverse)

    def run_raw(self, raws: Sequence[np.ndarray], windows, reverse: Sequence[Optional[bool]],
                spike_removal: Optional[str] = None, offset: float = 0.35) -> list:
        """``get_workload`` + ``run`` for reads still in DAC counts (wrapper.py:44-54, 104-120): normalised
        and called on the device in one chain, order preserved.  ``windows=None``: each read's STR window is
        first found in the whole read (``locate_raw``); a read whose window is not found comes back as a
        ``caller.NotLocated`` instead of a CallerResult, and the windows are in ``engine.last_located``.  There
        a strand may be None: the read is searched on both strands and called on the one found
        (``caller.choose_strand``); ``engine.last_located['strand']`` has every read's strand (0 template,
        1 reverse, -1 found on neither).  Given windows need given strands (ValueError naming the read)."""
        return self._run(self.engine.call_raw_batch, raws, windows, reverse, spike_removal, offset)

    def run_compressed(self, reads, windows, reverse: Sequence[Optional[bool]],
                       spike_removal: Optional[str] = None, offset: float = 0.35) -> list:
        """``run_raw`` for reads as their fast5 files store them (fast5.CompressedRead, see
        ``get_compressed_workload``): the VBZ decode happens on the device too, order preserved.  None strands
        as in ``run_raw``."""
        return self._run(self.engine.call_vbz_batch, reads, windows, reverse, spike_removal, offset)

    def _run(self, call, reads, windows, reverse, spike_removal, offset) -> list:
        """``run_raw`` with the engine's ``call`` of the reads' form; errors name a read by its name, else '#k'."""
        reverse = _strands(reverse)
        if windows is not None:
            _need_strands(reverse, [getattr(r, 'read_name', f'#{k}') for k, r in enumerate(reads)], 'a given window')
        return call(reads, windows, self._aut(reverse), reverse, spike_removal or self.caller_config.spike_removal,
                    offset)

    def _aut(self, reverse):
        """Per read the automaton of its strand, or the (template, reverse) pair where the strand is None."""
        return [(self._temp_id, self._rev_id) if rv is None else self._rev_id if rv else self._temp_id
                for rv in reverse]

    # -- STR windows without a basecall (DESIGN.md section 4.5) ----------------------------------------------
    def locate_raw(self, raws: Sequence[np.ndarray], reverse: Sequence[Optional[bool]],
                   spike_removal: Optional[str] = None, offset: float = 0.35) -> dict:
        """The STR window ``[lo, hi]`` of every whole raw read, found by searching the strand's automaton
        (flank - repeat - flank) in the whole normalised read: host arrays ``lo``, ``hi``, ``score`` and
        ``status`` (0 found, 1 nothing scores below zero, 2 the read is too short).  A read whose strand is None
        is searched on both strands and ``caller.choose_strand`` picks one; ``strand`` holds every read's strand
        (0 template, 1 reverse, given or detected; -1 found on neither), ``strand_score`` / ``strand_status`` /
        ``strand_lo`` / ``strand_hi`` (n, 2) both searches of those reads (NaN / -1 for a read with a given
        strand)."""
        return self._locate(_WholeReads(*pack_raw(raws)) if raws else None, reverse, spike_removal, offset)

    def locate_compressed(self, reads, reverse: Sequence[Optional[bool]], spike_removal: Optional[str] = None,
                          offset: float = 0.35) -> dict:
        """``locate_raw`` for reads as their fast5 files store them (fast5.CompressedRead): decoded on the device.
        A chunk the host decoder would refuse raises that Fast5FormatError."""
        return self._locate(_VBZReads(*pack_vbz(reads), reads) if reads else None, reverse, spike_removal, offset)

    def _locate(self, src, reverse, spike_removal, offset) -> dict:
        """``locate_raw`` of whole reads in any form (a ``caller._WholeReads``; None: no reads)."""
        reverse = _strands(reverse)
        if src is None:
            return _no_reads()
        res = self.engine._locate_whole(src, self._aut(reverse), spike_removal or self.caller_config.spike_removal,
                                        offset)
        src.raise_bad(res)
        fill_given_strands(res, reverse)
        return res

    # -- state similarity report (wrapper.py:122-160) ------------------------------------------------
    def check_high_similarity(self, sequence: str):
        diffs = {'template': self.pore_model.get_diffs_for_all(sequence),
                 'reverse': self.pore_model.get_diffs_for_all(self.reverse_uniq_sequence(sequence))}
        out_path = os.path.join(self.locus.path, tmpl.SUMMARY_SUBDIR, 'state_similarity.csv')
        try:
            with open(out_path, 'w') as fh:
                fh.write('pattern,strand,mean_diff,median_diff\n')
                for strand, table in diffs.items():
                    for pat, (mean_d, med_d) in table.items():
                        fh.write(f'{pat},{strand},{mean_d:.3f},{med_d:.3f}\n')
        except OSError:
            pass
        limit = self.caller_config.min_state_similarity
        problems = {strand: [dict(pattern=pat, mean_diff=v[0], median_diff=v[1])
                             for pat, v in table.items() if limit > v[0] or limit > v[1]]
                    for strand, table in diffs.items()}
        for p in problems['template']:
            print('Warning: Template has repeat unit {} with high state similarity'.format(p['pattern']))
        for p in problems['reverse']:
            print('Warning: high similarity of state values in reverse pattern {}'.format(p['pattern']))
        return problems['template'], problems['reverse']

    # -- complex loci (wrapper.py:162-248) -----------------------------------------------------------
    def break_into_units(self, template: str):
        """Top-level bracketed groups of the locus regex, the plain-base strings each can emit
        per loop iteration, and the number of unbracketed bases in front of each group."""
        opened: List[int] = []
        units: List[str] = []
        offsets: List[int] = []
        plain = 0
        for pos, ch in enumerate(template):
            if ch in '({':
                opened.append(pos)
            elif ch in ')}':
                begin = opened.pop()
                if not opened:
                    units.append(template[begin:pos + 1])
                    offsets.append(plain)
                    plain = 0
            elif not opened:
                plain += 1

        repeat_units: List[List[str]] = []
        for unit in units:
            variants: List[str] = []
            cur = ''
            for ch in unit:
                if ch in '()':
                    continue
                if ch == '{':
                    variants.append(cur)
                    cur = ''
                elif ch == '}':
                    variants.extend([v + cur for v in list(variants)])
                    cur = ''
                else:
                    cur += ch
            if cur:
                variants.append(cur)
            expanded: List[str] = []
            for var in variants:
                outs = ['']
                for ch in var:
                    if ch in tmpl.DNA_DICT:
                        outs = [o + alt for alt in tmpl.DNA_DICT[ch] for o in outs]
                    else:
                        outs = [o + ch for o in outs]
                expanded.extend(outs)
            repeat_units.append(expanded)
        return units, repeat_units, offsets

    def collapse_repeats(self, seq: str):
        """Counts of every repeat-unit variant in a called sequence (wrapper.py:220-248)."""
        results = [[0] * len(u) for u in self.repeat_units]
        rest = seq
        for n, (variants, off) in enumerate(zip(self.repeat_units, self.offsets)):
            rest = rest[off:]
            while rest:
                nxt = None
                for v, cand in enumerate(variants):
                    if cand == rest[:len(cand)]:
                        results[n][v] += 1
                        nxt = rest[len(cand):]      # the last matching variant decides what is consumed
                if nxt is None:
                    break
                rest = nxt
        return results


def get_raw_workload(df_overview, path: str):
    """The saved reads of a locus as they are on disk: (names, reverse flags, raw int16 signals, windows; a
    window is None where the row leaves it empty).
    The raw signal of every saved read comes from its annotated single-read fast5
    (``<locus>/fast5/<run_id>/annot/<read>.fast5``, what the reference's extraction step
    writes) or, for a caller-only run prepared straight from a sequencing run's multi-read
    files, from the file named in the row's ``fast5_path`` column, a multi-read fast5 or a POD5 file (see
    caller_only.py)."""
    from .fast5 import raw_signal
    names, revs, raws, wins = [], [], [], []
    has_src = 'fast5_path' in df_overview.columns
    for row in df_overview.itertuples():
        if row.saved:
            raws.append(raw_signal(*_read_source(row, path, has_src)))
            names.append(row.Index)
            revs.append(_strand(row))
            wins.append(_window(row))
    return names, revs, raws, wins


def _strands(reverse) -> list:
    """Strand flags as bools, None kept (a strand to be found)."""
    return [None if r is None else bool(r) for r in reverse]


def _need_strands(reverse, names, what: str) -> None:
    missing = [str(n) for n, r in zip(names, reverse) if r is None]
    if missing:
        raise ValueError(f'read {missing[0]}: {what} needs a strand (reverse), and none is given'
                         + (f' (nor for {len(missing) - 1} more)' if len(missing) > 1 else ''))


def _no_reads() -> dict:
    return dict(lo=np.zeros(0, np.int32), hi=np.zeros(0, np.int32), score=np.zeros(0), status=np.zeros(0, np.int32),
                strand=np.zeros(0, np.int8), strand_score=np.zeros((0, 2)), strand_status=np.zeros((0, 2), np.int32),
                strand_lo=np.zeros((0, 2), np.int32), strand_hi=np.zeros((0, 2), np.int32))


def _strand(row) -> Optional[bool]:
    """``reverse`` of an overview row, or None where the row leaves it empty (caller_only.py): the strand is
    then found in the whole read.  pandas reads a column of True, False and empty cells as bools and NaN; a cell
    read as text (a column with other values) is parsed, never passed to bool(), for which 'False' is true."""
    v = row.reverse
    if isinstance(v, str):
        t = v.strip().lower()
        if t in ('true', 'false', ''):
            return None if t == '' else t == 'true'
        raise ValueError(f'read {row.Index}: reverse must be True, False or empty, not {v!r}')
    if pd.isna(v):
        return None
    return bool(v)


def _window(row):
    """(l_start_raw, r_end_raw) of an overview row, or None where the row leaves them empty (caller_only.py)."""
    if pd.isna(row.l_start_raw) or pd.isna(row.r_end_raw):
        return None
    return int(row.l_start_raw), int(row.r_end_raw)


def _read_source(row, path: str, has_src: bool):
    """(file, read name or None) a saved overview row's signal comes from: its annotated single-read fast5,
    else the multi-read fast5 or POD5 file of the row's ``fast5_path``."""
    fpath = os.path.join(path, tmpl.FAST5_SUBDIR, str(row.run_id), tmpl.ANNOT_SUBDIR, row.Index + '.fast5')
    if os.path.exists(fpath):
        return fpath, None
    if has_src and isinstance(row.fast5_path, str) and os.path.exists(row.fast5_path):
        return row.fast5_path, row.Index
    raise FileNotFoundError(f'no fast5 for read {row.Index}: {fpath}')


def get_compressed_workload(df_overview, path: str):
    """``get_raw_workload`` without the host's StreamVByte decode: (names, reverse flags, reads as their
    files store them (fast5.CompressedRead from ``fast5.stored_chunks``: zstd frames left for the GPU too,
    the others undone on the host), windows).  Files are found as ``get_raw_workload`` finds them, and each is
    opened and parsed once for all its rows, fast5 or POD5 alike (``fast5.open_raw``)."""
    from .fast5 import open_raw, stored_chunks
    names, revs, reads, wins = [], [], [], []
    has_src = 'fast5_path' in df_overview.columns
    rows = [row for row in df_overview.itertuples() if row.saved]
    sources = [_read_source(row, path, has_src) for row in rows]
    by_file = {}
    for k, (fpath, _) in enumerate(sources):
        by_file.setdefault(fpath, []).append(k)
    reads = [None] * len(rows)
    for fpath, ks in by_file.items():
        with open_raw(fpath) as f:
            for k in ks:
                reads[k] = stored_chunks(fpath, sources[k][1], f)
    for row in rows:
        names.append(row.Index)
        revs.append(_strand(row))
        wins.append(_window(row))
    return names, revs, reads, wins


def get_workload(df_overview, path: str, spike_removal: str = 'Brute') -> List[ReadSignal]:
    """Reads of the locus with their normalised STR windows (reference: wrapper.py:44-54): all reads are
    spike-filtered, MAD normalised and sliced in one GPU launch and returned as host float64 arrays, which
    is what the reference's ``ReadSignal`` holds.  ``main_wrapper`` does not take this detour: it hands the
    compressed reads to ``CallerWrapper.run_compressed``, which decodes them and keeps the windows on the device."""
    from .normalize import normalize_windows
    names, revs, raws, wins = get_raw_workload(df_overview, path)
    sigs = normalize_windows(raws, wins, spike_removal)
    return [ReadSignal(n, r, s) for n, r, s in zip(names, revs, sigs)]


def _run_locating(call_wrapper, df_overview, names, revs, reads, wins, spike_removal, offset):
    """main_wrapper's call of a locus where some rows leave their window empty: those reads are located in
    the whole read first (on both strands where ``reverse`` is empty too) and their windows, and detected
    strands, are written into the overview's columns; a read whose window is not found gets no result (a
    caller.NotLocated) and keeps its empty cells, and all such reads are named in one warning.  Returns the
    results and the strands (detected ones filled in; None for a read found on neither)."""
    import warnings
    results = [None] * len(reads)
    revs = list(revs)
    given = [k for k, w in enumerate(wins) if w is not None]
    missing = [k for k, w in enumerate(wins) if w is None]
    if given:
        for k, r in zip(given, call_wrapper.run_compressed([reads[k] for k in given], [wins[k] for k in given],
                                                           [revs[k] for k in given], spike_removal)):
            results[k] = r
    located = call_wrapper.run_compressed([reads[k] for k in missing], None, [revs[k] for k in missing],
                                          spike_removal, offset)
    loc = call_wrapper.engine.last_located
    lo = df_overview['l_start_raw'].astype('Int64')
    hi = df_overview['r_end_raw'].astype('Int64')
    detect = any(revs[k] is None for k in missing)
    strand = df_overview['reverse'].astype(object) if detect else None
    lost = []
    for i, (k, r) in enumerate(zip(missing, located)):
        results[k] = r
        if loc['status'][i] == 0:
            lo[names[k]] = int(loc['lo'][i])
            hi[names[k]] = int(loc['hi'][i])
            if revs[k] is None:
                revs[k] = bool(loc['strand'][i] == 1)
                strand[names[k]] = revs[k]
        else:
            lost.append(names[k])
    df_overview['l_start_raw'] = lo
    df_overview['r_end_raw'] = hi
    if detect:
        df_overview['reverse'] = strand
    if lost:
        warnings.warn(f'{len(lost)} read(s) without a window in the overview: the STR window was not found in the '
                      f'whole read, so they have no result: {", ".join(map(str, lost))}', RuntimeWarning, stacklevel=3)
    return results, revs


def main_wrapper(locus: Locus, threads: int = 1, config: Optional[Config] = None,
                 workload: Optional[Sequence[ReadSignal]] = None, flanks: Optional[Flanks] = None,
                 engine: Optional[CallerEngine] = None, offset: float = 0.35):
    """The caller step of one locus (reference: wrapper.py:17-41): overview.csv in, calls on the
    GPU, overview.csv / FASTA / complex-unit CSV out.  Plots are not produced.  ``workload``
    (one ReadSignal per saved overview row, in row order) bypasses the fast5 reading.  Rows whose
    ``l_start_raw`` / ``r_end_raw`` are empty are located in the whole read first (DESIGN.md section 4.5,
    score offset ``offset``) and get the located window written into those columns; rows whose ``reverse`` is
    empty as well are searched on both strands and get the detected strand written into ``reverse`` (so the
    FASTA files and the complex-unit CSV split on it); rows whose window is not found keep empty result columns.
    A row with a window but no strand raises ValueError."""
    from .overview import load_overview, store_collapsed, store_results
    overview_path, df_overview = load_overview(locus.path)
    cc = config.caller_config if config is not None else CallerConfig()
    call_wrapper = CallerWrapper(locus, threads, flanks=flanks, config=config, engine=engine)
    if workload is None:
        # the reads' VBZ chunks as stored -> zstd decode -> StreamVByte decode -> normalisation kernel -> caller,
        # all on the device
        names, revs, reads, wins = get_compressed_workload(df_overview, locus.path)
        if all(w is not None for w in wins):
            results = call_wrapper.run_compressed(reads, wins, revs, cc.spike_removal)
        else:
            results, revs = _run_locating(call_wrapper, df_overview, names, revs, reads, wins, cc.spike_removal,
                                          offset)
        workload = [ReadSignal(n, r, None) for n, r in zip(names, revs)]
    else:
        results = call_wrapper.run(workload)
    seq_results = [(r.seq, r.resc_seq) if isinstance(r, CallerResult) else None for r in results]
    cost_results = [(r.cost, r.resc_cost) if isinstance(r, CallerResult) else None for r in results]
    df_overview = store_results(overview_path, df_overview, seq_results, cost_results, locus.path)
    df_collapsed = None
    if len(call_wrapper.units) > 1:
        print(f'Running complex genotyping as complex repeat units present: {call_wrapper.units}')
        called = [k for k, sr in enumerate(seq_results) if sr is not None]
        workload = [workload[k] for k in called]
        collapsed = [call_wrapper.collapse_repeats(seq_results[k][1]) for k in called]
        df_collapsed = store_collapsed(collapsed, call_wrapper.units, call_wrapper.repeat_units,
                                       [bool(r.reverse) for r in workload], locus.path)
    return df_overview, df_collapsed
