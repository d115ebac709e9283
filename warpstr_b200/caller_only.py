"""Caller-only preparation (reference: prepare_caller_only.py at the repository root).

The reference takes a CSV with ``fast5_path, locus, read_name, reverse, l_start_raw,
r_end_raw`` (optionally ``run_id``), copies every read out of its multi-read fast5 into a
single-read file under ``<output>/<locus>/fast5/<run_id>/annot/`` (h5py) and writes
``<output>/<locus>/overview.csv``.  This build cannot write HDF5 and does not need to: the
overview keeps the ``fast5_path`` column (the reference keeps it too) and
``wrapper.get_workload`` reads the signal straight from the multi-read file.

The STR window columns ``l_start_raw, r_end_raw`` may be left out, or left empty in some rows: the
caller then finds those reads' windows itself in the whole read (``wrapper.main_wrapper``, DESIGN.md
section 4.5).  The ``reverse`` column is required but its cells may be empty too: such a read is searched
on both strands and the strand found is written into the overview.  So the run's fast5 files and the
names of a locus's reads are enough, e.g. read IDs of targeted or adaptive sampling, which come without
strands.  A window is only taken with its strand: a row with a window and an empty ``reverse`` is refused.

    python -m warpstr_b200.caller_only --config cfg.yaml --file reads.csv
"""
import argparse
import csv
import os
from typing import Dict, List

import yaml

from . import fast5

REQUIRED = ['fast5_path', 'locus', 'read_name', 'reverse']
WINDOW = ['l_start_raw', 'r_end_raw']       # optional; an overview always gets them, empty where not given


def prepare(output: str, csv_path: str, check_reads: bool = True) -> Dict[str, str]:
    """Write ``<output>/<locus>/overview.csv`` for every locus of the CSV; returns
    {locus: overview path}.  Errors match the reference script's."""
    if not os.path.exists(csv_path):
        raise FileNotFoundError(f'CSV File={csv_path} does not exists')
    with open(csv_path, 'r') as fh:
        reader = csv.reader(fh)
        header = next(reader)
        if any(col not in REQUIRED + WINDOW + ['run_id'] for col in header) or any(col not in header for col in REQUIRED):
            raise ValueError(f'Not all required columns present in input CSV file. Required fields are: {REQUIRED}, '
                             f'optional: {WINDOW + ["run_id"]}')
        add_win = [c for c in WINDOW if c not in header]
        add_run_id = 'run_id' not in header
        rows: Dict[str, List[List[str]]] = {}
        known: Dict[str, set] = {}
        for row in reader:
            if not row:
                continue
            rec = dict(zip(header, row))
            if not rec.get('reverse', '').strip() and any(rec.get(c, '').strip() for c in WINDOW):
                raise ValueError(f"Read {rec['read_name']}: a window (l_start_raw, r_end_raw) is given without "
                                 f"its strand (reverse is empty)")
            if check_reads:
                src = rec['fast5_path']
                if src not in known:
                    known[src] = set(fast5.read_names(src))
                if rec['read_name'] not in known[src]:
                    raise ValueError(f"Read {rec['read_name']} not found in fast5 file {src}")
            rows.setdefault(rec['locus'], []).append(row + [''] * len(add_win) + (['run_0'] if add_run_id else []) +
                                                     ['1'])
    out_header = header + add_win + (['run_id'] if add_run_id else []) + ['saved']
    written = {}
    for locus, lines in rows.items():
        dest = os.path.join(output, locus)
        os.makedirs(dest, exist_ok=True)
        path = os.path.join(dest, 'overview.csv')
        with open(path, 'w') as fh:
            w = csv.writer(fh, delimiter=',', quotechar='"', quoting=csv.QUOTE_MINIMAL)
            w.writerow(out_header)
            w.writerows(lines)
        written[locus] = path
    return written


def main(argv=None):
    ap = argparse.ArgumentParser(description='WarpSTR caller-only preparation')
    ap.add_argument('--config', required=True, help='input config')
    ap.add_argument('--file', required=True, help='csv file')
    args = ap.parse_args(argv)
    if not os.path.exists(args.config):
        raise FileNotFoundError(f'Config File={args.config} does not exists')
    with open(args.config, 'r') as fh:
        config = yaml.safe_load(fh)
    written = prepare(config['output'], args.file)
    print(f'Finished preparing WarpSTR document structure for the input config {args.config} and csv file {args.file}')
    for locus, path in written.items():
        print(f'  {locus}: {path}')


if __name__ == '__main__':
    main()
