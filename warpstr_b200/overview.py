"""Result files of the caller step: ``overview.csv`` columns, FASTA files, complex-unit CSV.

Same file contract as the reference's caller/overview.py (the genotyper and the user read
these): ``results`` = len(resc_seq), ``orig`` = len(seq), ``dtw_cost1/2`` (:57-73, 103-115),
``predictions/sequences/{all,sequences_template,sequences_reverse}.fasta`` (:76-100) and
``predictions/complexSTR_analysis/complex_repeat_units.csv`` (:11-34).
"""
import os
from typing import List, Sequence, Tuple

import numpy as np
import pandas as pd

from . import templates as tmpl


def load_overview(locus_path: str):
    overview_path = os.path.join(locus_path, tmpl.OVERVIEW_NAME)
    try:
        df = pd.read_csv(overview_path)
    except FileNotFoundError:
        raise FileNotFoundError(f'Not found the overview file {overview_path} - Please check the "output" in config')
    df.set_index('read_name', inplace=True)
    df.columns = df.columns.map(str)
    return overview_path, df


def append_results(seq_results: Sequence[Tuple[str, str]], cost_results: Sequence[Tuple[float, float]], df):
    """One entry per overview row; rows that were not extracted (``saved`` false) get -1, saved rows without a
    result (``None`` in ``seq_results``: the STR window was not found) get None."""
    fasta, results, orig, c1, c2 = [], [], [], [], []
    k = 0
    for row in df.itertuples():
        if row.saved and seq_results[k] is None:
            for col in (results, orig, c1, c2):
                col.append(None)
            k += 1
        elif row.saved:
            seq, resc = seq_results[k]
            results.append(len(resc))
            orig.append(len(seq))
            c1.append(cost_results[k][0])
            c2.append(cost_results[k][1])
            fasta.append((row.Index, resc, row.reverse))
            k += 1
        else:
            results.append(-1)
            orig.append(-1)
            c1.append(-1)
            c2.append(-1)
    return fasta, results, orig, c1, c2


def write_results_to_fasta(fasta: List[Tuple[str, str, bool]], locus_path: str) -> None:
    out_dir = os.path.join(locus_path, tmpl.PREDICTIONS_SUBDIR, 'sequences')
    os.makedirs(out_dir, exist_ok=True)

    def dump(name, keep):
        with open(os.path.join(out_dir, name), 'w') as fh:
            for read_id, seq, rev in fasta:
                if keep(rev):
                    fh.write(f'>{read_id}\n{seq}\n\n')

    dump('all.fasta', lambda rev: True)
    dump('sequences_template.fasta', lambda rev: rev is False or rev is np.False_)
    dump('sequences_reverse.fasta', lambda rev: bool(rev))


def save_overview(overview_path: str, df, results, orig, c1, c2):
    old = [c for c in df.columns if c.startswith('result')]
    df.drop(columns=old, inplace=True)
    if any(r is None for r in results):    # rows without a result: empty cells, the other lengths still integers
        results, orig = pd.array(results, dtype='Int64'), pd.array(orig, dtype='Int64')
        c1, c2 = pd.array(c1, dtype='Float64'), pd.array(c2, dtype='Float64')
    df['results'] = results
    df['orig'] = orig
    df['dtw_cost1'] = c1
    df['dtw_cost2'] = c2
    df.to_csv(overview_path)
    print(f' Results stored in overview file {overview_path}')
    return df


def store_results(overview_path: str, df, seq_results, cost_results, locus_path: str):
    fasta, results, orig, c1, c2 = append_results(seq_results, cost_results, df)
    write_results_to_fasta(fasta, locus_path)
    return save_overview(overview_path, df, results, orig, c1, c2)


def store_collapsed(results, units: List[str], rep_units: List[List[str]], reverse_lst: List[bool], locus_path: str):
    """Per-read repeat-unit counts of a complex locus (reference: overview.py:11-34)."""
    cols = {}
    for n, unit in enumerate(units):
        if len(results[0][n]) > 1:
            cols['main_' + rep_units[n][0]] = np.array([np.sum(r[n]) for r in results])
            for v, variant in enumerate(rep_units[n][1:]):
                cols['inter_' + variant[len(rep_units[n][0]):]] = np.array([r[n][v + 1] for r in results])
        else:
            cols[unit.strip('(').strip(')')] = np.array([r[n][0] for r in results])
    cols['reverse'] = reverse_lst
    df = pd.DataFrame.from_dict(cols)
    out_dir = os.path.join(locus_path, tmpl.PREDICTIONS_SUBDIR, tmpl.COMPLEX_SUBDIR)
    os.makedirs(out_dir, exist_ok=True)
    df.to_csv(os.path.join(out_dir, 'complex_repeat_units.csv'))
    return df
