"""A panel's reads found in a whole run by their flanks (DESIGN.md section 4.6).

The caller needs to know which reads belong to which locus.  Usually that comes from a basecall and an alignment
(a BAM), listed in the CSV ``caller_only.prepare`` takes.  Here it comes from the raw signal itself: each locus's
flanks are unique sequence, so every read of the run is searched for them on the GPU, and a read whose two
flanks of one strand are found, in order, belongs to that locus on that strand.  The repeat between the flanks
plays no part: a long expansion of the same motif at another locus, or any genomic run of it, matches a repeat
automaton well enough to outweigh two poorly matched flanks, but cannot make a flank match.

Each locus gets four chain automata (``StateAutomata`` of a sequence without loops): the template strand's left
and right flank and the reverse strand's left and right flank, in that order (``CHAINS``).  They are searched with
the window search of DESIGN.md section 4.5 (score offset 0.35 per sample), all of a panel's chains in one launch
(wstr_assign_batch), and ``choose_loci`` is the rule applied to the four searches of a (read, locus).

``assign_files`` goes from ``.fast5`` / ``.pod5`` files and a config to ``<output>/<locus>/overview.csv``, one row
per read found with its detected strand and empty window cells; ``wrapper.main_wrapper`` then finds each read's
window itself (section 4.5) and calls it.

    python -m warpstr_b200.assign --config cfg.yaml RUN [RUN ...]

Each RUN is a ``.fast5`` / ``.pod5`` file or a directory searched (recursively) for them.
"""
import argparse
import os
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib, fast5
from .automata import StateAutomata
from .caller import HIT_FIELDS
from .caller_only import write_overviews
from .config import Config, load_config
from .pore_model import PoreModel, get_pore_model
from .wrapper import Flanks, load_flanks

CHAINS = ('template_left', 'template_right', 'reverse_left', 'reverse_right')
OVERVIEW_HEADER = ['fast5_path', 'locus', 'read_name', 'reverse', 'l_start_raw', 'r_end_raw', 'run_id', 'saved']
RAW_SUFFIXES = ('.fast5', '.pod5')


def flank_chains(flanks: Flanks, pore_model: Optional[PoreModel] = None) -> List[StateAutomata]:
    """The four chain automata of one locus, in ``CHAINS`` order."""
    pm = pore_model or get_pore_model()
    return [StateAutomata(s, pm) for s in (flanks.template.left, flanks.template.right, flanks.reverse.left,
                                           flanks.reverse.right)]


class Panel:
    """Every locus of a panel, in order, with its four flank chains (``chains[4 * k : 4 * k + 4]`` are locus k's).
    ``register(engine)`` uploads the chains to an engine once and gives their automaton ids there."""

    def __init__(self, loci: Sequence[Tuple[str, Flanks]], min_values_per_state: int = 4, flank_length: int = 110,
                 pore_model: Optional[PoreModel] = None):
        if not loci:
            raise ValueError('a panel needs at least one locus')
        self.names = [name for name, _ in loci]
        self.chains = [c for _, f in loci for c in flank_chains(f, pore_model)]
        self.min_values_per_state = int(min_values_per_state)
        self.flank_length = int(flank_length)
        self._ids = weakref.WeakKeyDictionary()

    @classmethod
    def from_config(cls, config: Config, flanks: Optional[Dict[str, Flanks]] = None,
                    pore_model: Optional[PoreModel] = None) -> 'Panel':
        """Every locus of ``config`` in config order; its flanks from ``flanks[name]`` or, by default, from the
        file the locus step writes under ``<output>/<locus>`` (``wrapper.load_flanks``)."""
        loci = [(lc.name, flanks[lc.name] if flanks is not None else load_flanks(os.path.join(config.output, lc.name)))
                for lc in config.loci]
        return cls(loci, config.caller_config.min_values_per_state, config.flank_length, pore_model)

    def register(self, engine) -> List[int]:
        ids = self._ids.get(engine)
        if ids is None:
            if engine.cc.min_values_per_state != self.min_values_per_state:
                raise ValueError(f'the panel was built for min_values_per_state {self.min_values_per_state}, the '
                                 f'engine calls with {engine.cc.min_values_per_state}')
            ids = [engine.add_automaton(c, self.flank_length) for c in self.chains]
            self._ids[engine] = ids
        return ids


def choose_loci(lo, hi, score, status) -> Dict[str, np.ndarray]:
    """The decision rule of the assignment, on the searches of every (read, chain): arrays [n_reads, 4 * n_loci],
    chains in panel order.  Per (read, locus):

    * a strand passes iff both of its flank chains are _lib.LOCATE_FOUND and left.hi < right.lo;
    * one strand passing gives that strand; both passing give the lower left.score + right.score, an exact tie the
      template (as ``caller.choose_strand``);
    * a read passing for several loci is assigned to each of them.

    Returns the hits, one array per field of ``caller.HIT_FIELDS``, sorted by (read, locus): the chosen strand
    (0 template, 1 reverse) and its two flanks' windows and scores.  wstr_assign_batch applies the same rule on
    the device."""
    status = np.asarray(status)
    shape = (status.shape[0], status.shape[1] // 4, 4)
    lo, hi, status = (np.asarray(a, dtype=np.int32).reshape(shape) for a in (lo, hi, status))
    score = np.asarray(score, dtype=np.float64).reshape(shape)
    found = status == _lib.LOCATE_FOUND
    t = found[..., 0] & found[..., 1] & (hi[..., 0] < lo[..., 1])
    r = found[..., 2] & found[..., 3] & (hi[..., 2] < lo[..., 3])
    rev = np.where(t & r, score[..., 2] + score[..., 3] < score[..., 0] + score[..., 1], r)
    read, locus = np.nonzero(t | r)
    strand = rev[read, locus].astype(np.int32)
    a = 2 * strand
    return dict(read=read.astype(np.int32), locus=locus.astype(np.int32), strand=strand,
                left_lo=lo[read, locus, a], left_hi=hi[read, locus, a], left_score=score[read, locus, a],
                right_lo=lo[read, locus, a + 1], right_hi=hi[read, locus, a + 1], right_score=score[read, locus, a + 1])


def scan_runs(runs: Sequence[str]) -> List[str]:
    """The raw-signal files of ``runs``: a file is taken as it is, a directory is searched recursively for
    ``.fast5`` / ``.pod5`` files (sorted, so the order is the same on every file system).  Each file once, in
    order."""
    out: List[str] = []
    for run in runs:
        if os.path.isdir(run):
            for root, dirs, files in os.walk(run):
                dirs.sort()
                out += [os.path.join(root, f) for f in sorted(files) if f.lower().endswith(RAW_SUFFIXES)]
        elif os.path.isfile(run):
            out.append(run)
        else:
            raise FileNotFoundError(f'{run} is neither a file nor a directory')
    return list(dict.fromkeys(out))


def assign_files(config: Config, files: Sequence[str], engine=None, flanks: Optional[Dict[str, Flanks]] = None,
                 chunk_reads: int = 4000, offset: float = 0.35, verbose: bool = True) -> Dict[str, int]:
    """Every read of ``files`` (multi-read fast5 or POD5, ``fast5.open_raw``) searched for the flanks of every
    locus of ``config`` (``Panel.from_config``; ``flanks`` as there), and ``<output>/<locus>/overview.csv`` written
    for each locus with reads: columns ``OVERVIEW_HEADER``, the detected strand in ``reverse``, the window cells
    empty; rows in file order, a file's reads in read-ID order, so a run gives the same overview from fast5 and from
    POD5.  The reads go to the device ``chunk_reads`` at a time as their files store them (zstd and VBZ decoded
    there, ``CallerEngine.assign_arrays_vbz``), so the buffers stay the same size whatever the run's.  Prints one
    line per locus and returns {locus: reads assigned}."""
    from .caller import CallerEngine, pack_vbz
    panel = Panel.from_config(config, flanks)
    if engine is None:
        engine = CallerEngine(config.caller_config, config.rescaler_config)
    rows: Dict[str, List[List[str]]] = {name: [] for name in panel.names}
    batch: list = []

    def flush():
        if not batch:
            return
        res = engine.assign_arrays_vbz(*pack_vbz(batch), panel, config.caller_config.spike_removal, offset,
                                       reads=batch)
        for r, k, s in zip(res['read'].tolist(), res['locus'].tolist(), res['strand'].tolist()):
            rows[panel.names[k]].append([batch[r].path, panel.names[k], batch[r].read_name, str(bool(s)), '', '',
                                         'run_0', '1'])
        batch.clear()

    for path in files:
        with fast5.open_raw(path) as f:
            for name in sorted(f.read_names()):
                read = fast5.stored_chunks(path, name, h5=f)
                if read.n_samples > 0:
                    batch.append(read)
                if len(batch) >= chunk_reads:
                    flush()
    flush()
    write_overviews(config.output, OVERVIEW_HEADER, {k: v for k, v in rows.items() if v})
    counts = {k: len(v) for k, v in rows.items()}
    if verbose:
        for k, c in counts.items():
            print(f'{k}: {c} reads assigned')
    return counts


def main(argv=None):
    ap = argparse.ArgumentParser(description='WarpSTR: find the reads of every locus of a config in raw-signal files '
                                             'by their flanks, and write each locus\'s overview.csv')
    ap.add_argument('--config', required=True, help='input config (YAML)')
    ap.add_argument('runs', nargs='+', metavar='RUN', help='a .fast5 / .pod5 file, or a directory searched for them')
    args = ap.parse_args(argv)
    config = load_config(args.config)
    files = scan_runs(args.runs)
    if not files:
        raise FileNotFoundError(f'no .fast5 or .pod5 file in {" ".join(args.runs)}')
    return assign_files(config, files)


if __name__ == '__main__':
    main()
