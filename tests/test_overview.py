"""CPU: the caller step's file contract (overview.csv columns, FASTA, complex-unit CSV)."""
import json
import os

import numpy as np
import pandas as pd
import pytest

from warpstr_b200 import overview as ov


def _make_locus_dir(tmp_path):
    d = tmp_path / 'LOC'
    d.mkdir()
    df = pd.DataFrame({'read_name': ['r1', 'r2', 'r3', 'r4'], 'run_id': ['a', 'a', 'b', 'b'],
                       'reverse': [False, True, False, True], 'saved': [1, 0, 1, 1],
                       'l_start_raw': [10, 20, 30, 40], 'r_end_raw': [500, 600, 700, 800],
                       'results': [9, 9, 9, 9], 'result_old': [1, 2, 3, 4]})
    df.to_csv(d / 'overview.csv', index=False)
    return str(d)


SEQS = [('AGCAGC', 'AGCAGCAGC'), ('CGC', 'CGCCGC'), ('A', '')]
COSTS = [(0.11, 0.09), (0.2, 0.19), (0.3, float('nan'))]


def test_store_results_contract(tmp_path):
    path = _make_locus_dir(tmp_path)
    ovp, df = ov.load_overview(path)
    out = ov.store_results(ovp, df, SEQS, COSTS, path)
    assert list(out['results']) == [9, -1, 6, 0] and list(out['orig']) == [6, -1, 3, 1]
    assert 'result_old' not in out.columns and out.loc['r2', 'dtw_cost1'] == -1
    back = pd.read_csv(ovp)
    assert list(back.columns[:1]) == ['read_name'] and {'results', 'orig', 'dtw_cost1', 'dtw_cost2'} <= set(back.columns)
    seqdir = os.path.join(path, 'predictions', 'sequences')
    assert open(os.path.join(seqdir, 'all.fasta')).read() == '>r1\nAGCAGCAGC\n\n>r3\nCGCCGC\n\n>r4\n\n\n'
    assert open(os.path.join(seqdir, 'sequences_template.fasta')).read() == '>r1\nAGCAGCAGC\n\n>r3\nCGCCGC\n\n'
    assert open(os.path.join(seqdir, 'sequences_reverse.fasta')).read() == '>r4\n\n\n'


def test_store_collapsed_contract(tmp_path):
    units = ['((CAGG){CAGM})', '(CAGA)', '(CA)']
    reps = [['CAGG', 'CAGGCAGA', 'CAGGCAGC'], ['CAGA'], ['CA']]
    results = [[[3, 1, 0], [2], [5]], [[4, 0, 2], [1], [7]]]
    df = ov.store_collapsed(results, units, reps, [False, True], str(tmp_path))
    assert list(df.columns) == ['main_CAGG', 'inter_CAGA', 'inter_CAGC', 'CAGA', 'CA', 'reverse']
    assert list(df['main_CAGG']) == [4, 6] and list(df['inter_CAGC']) == [0, 2]
    assert os.path.exists(os.path.join(str(tmp_path), 'predictions', 'complexSTR_analysis', 'complex_repeat_units.csv'))


def test_missing_overview(tmp_path):
    with pytest.raises(FileNotFoundError):
        ov.load_overview(str(tmp_path))


def test_files_identical_to_the_reference(tmp_path):
    """The files the reference's store_results wrote for the same inputs (stored in
    golden/reference_pin.npz, see tests/test_reference_pin.py)."""
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_pin.npz'))
    want = json.loads(str(z['cases']))['overview_files']
    a = _make_locus_dir(tmp_path)
    os.makedirs(os.path.join(a, 'predictions', 'sequences'))
    ovp, df = ov.load_overview(a)
    ov.store_results(ovp, df, SEQS, COSTS, a)
    assert len(want) == 4
    for rel, text in want.items():
        assert open(os.path.join(a, rel)).read() == text, rel
