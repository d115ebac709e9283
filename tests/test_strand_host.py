"""CPU: reads without a strand (DESIGN.md section 4.5).  caller_only.prepare takes empty ``reverse`` cells and
refuses a window without its strand; an overview's mixed True / False / empty ``reverse`` column reads back as
bools and None; caller.choose_strand, the one decision rule between the two strands' searches."""
import csv
import os

import numpy as np
import pytest

from warpstr_b200 import _lib, caller_only
from warpstr_b200.caller import choose_strand, split_pairs
from warpstr_b200.overview import load_overview
from warpstr_b200.wrapper import _strand

F, NF, NP = _lib.LOCATE_FOUND, _lib.LOCATE_NOT_FOUND, _lib.LOCATE_NO_PATH
HEADER = ['fast5_path', 'locus', 'read_name', 'reverse', 'l_start_raw', 'r_end_raw']


def _write(tmp_path, header, rows):
    path = str(tmp_path / 'reads.csv')
    with open(path, 'w') as fh:
        fh.write(','.join(header) + '\n')
        for r in rows:
            fh.write(','.join(r) + '\n')
    return path


def test_prepare_takes_empty_strands(tmp_path):
    path = _write(tmp_path, HEADER, [['a.fast5', 'LOC', 'r1', '', '', ''], ['a.fast5', 'LOC', 'r2', 'True', '', ''],
                                     ['a.fast5', 'LOC', 'r3', 'False', '100', '900']])
    written = caller_only.prepare(str(tmp_path / 'out'), path, check_reads=False)
    with open(written['LOC']) as fh:
        rows = list(csv.DictReader(fh))
    assert [r['reverse'] for r in rows] == ['', 'True', 'False']
    assert [(r['l_start_raw'], r['r_end_raw']) for r in rows] == [('', ''), ('', ''), ('100', '900')]


def test_prepare_takes_empty_strands_without_window_columns(tmp_path):
    path = _write(tmp_path, HEADER[:4], [['a.fast5', 'LOC', 'r1', ''], ['a.fast5', 'LOC', 'r2', '']])
    written = caller_only.prepare(str(tmp_path / 'out'), path, check_reads=False)
    with open(written['LOC']) as fh:
        rows = list(csv.DictReader(fh))
    assert [r['reverse'] for r in rows] == ['', '']


@pytest.mark.parametrize('window', [('100', '900'), ('100', '')])
def test_prepare_refuses_a_window_without_strand(tmp_path, window):
    path = _write(tmp_path, HEADER, [['a.fast5', 'LOC', 'r1', 'True', '5', '50'],
                                     ['a.fast5', 'LOC', 'lonely', '', *window]])
    with pytest.raises(ValueError, match='lonely'):
        caller_only.prepare(str(tmp_path / 'out'), path, check_reads=False)
    assert not os.path.exists(str(tmp_path / 'out'))


def test_strand_of_overview_rows(tmp_path):
    path = _write(tmp_path, HEADER, [['a.fast5', 'LOC', 'r1', 'True', '', ''], ['a.fast5', 'LOC', 'r2', 'False', '', ''],
                                     ['a.fast5', 'LOC', 'r3', '', '', ''], ['a.fast5', 'LOC', 'r4', 'False', '', '']])
    written = caller_only.prepare(str(tmp_path / 'out'), path, check_reads=False)
    _, df = load_overview(os.path.dirname(written['LOC']))
    got = [_strand(row) for row in df.itertuples()]
    assert got == [True, False, None, False]
    assert all(g is None or type(g) is bool for g in got)


def test_strand_of_a_column_read_as_text():
    class Row:
        Index = 'r'

        def __init__(self, v):
            self.reverse = v
    assert [_strand(Row(v)) for v in ('True', 'False', 'false', ' ', np.nan, np.True_, 0.0)] == \
        [True, False, False, None, None, True, False]
    with pytest.raises(ValueError, match='r'):
        _strand(Row('maybe'))


def test_split_pairs():
    pair, ids = split_pairs([3, (0, 1), 1])
    assert pair.tolist() == [False, True, False]
    assert ids.tolist() == [[3, 3], [0, 1], [1, 1]]
    pair, ids = split_pairs(np.array([2, 5], dtype=np.int32))
    assert not pair.any() and ids.tolist() == [[2, 2], [5, 5]]


@pytest.mark.parametrize('status,score,strand,col,st,sc', [
    # found on one strand only: that strand, whatever the other's score
    ((F, NF), (-3.0, -9.0), 0, 0, F, -3.0),
    ((NF, F), (-9.0, -1.0), 1, 1, F, -1.0),
    ((NP, F), (np.inf, -2.0), 1, 1, F, -2.0),
    ((F, NP), (-2.0, np.inf), 0, 0, F, -2.0),
    # found on both: the lower score
    ((F, F), (-3.0, -7.5), 1, 1, F, -7.5),
    ((F, F), (-7.5, -3.0), 0, 0, F, -7.5),
    # exact tie: the template
    ((F, F), (-4.25, -4.25), 0, 0, F, -4.25),
    # neither: NOT_FOUND if either had it, else NO_PATH, and the lower score
    ((NF, NF), (2.0, 0.5), -1, 1, NF, 0.5),
    ((NF, NF), (0.0, 0.0), -1, 0, NF, 0.0),
    ((NF, NP), (3.0, np.inf), -1, 0, NF, 3.0),
    ((NP, NF), (np.inf, 3.0), -1, 1, NF, 3.0),
    ((NP, NF), (1.0, 3.0), -1, 0, NF, 1.0),
    ((NP, NP), (np.inf, np.inf), -1, 0, NP, np.inf),
])
def test_choose_strand(status, score, strand, col, st, sc):
    got = choose_strand(np.array([status]), np.array([score]))
    assert (int(got[0][0]), int(got[1][0]), int(got[2][0]), float(got[3][0])) == (strand, col, st, sc)
    assert got[0].dtype == np.int8 and got[2].dtype == np.int32


def test_choose_strand_batch_matches_rows():
    rng = np.random.default_rng(3)
    status = rng.integers(0, 3, size=(500, 2)).astype(np.int32)
    score = np.where(status == NP, np.inf, rng.integers(-4, 4, size=(500, 2)) / 2.0)
    strand, col, st, sc = choose_strand(status, score)
    for r in range(500):
        one = choose_strand(status[r:r + 1], score[r:r + 1])
        assert (strand[r], col[r], st[r], sc[r]) == tuple(x[0] for x in one)
    # a read given one strand is its own pair: status and score are that search's
    same = choose_strand(np.stack((status[:, 0], status[:, 0]), 1), np.stack((score[:, 0], score[:, 0]), 1))
    assert np.array_equal(same[2], status[:, 0]) and np.array_equal(same[3], score[:, 0]) and not same[1].any()
