"""CPU: caller_only.prepare takes a CSV whose STR window columns are missing or partly empty (the caller then
locates those windows itself) and still refuses one without ``reverse`` or ``read_name``."""
import csv
import os

import pytest

from warpstr_b200 import caller_only


def _prepare(tmp_path, header, rows):
    path = str(tmp_path / 'reads.csv')
    with open(path, 'w') as fh:
        fh.write(','.join(header) + '\n')
        for r in rows:
            fh.write(','.join(r) + '\n')
    written = caller_only.prepare(str(tmp_path / 'out'), path, check_reads=False)
    with open(written['LOC']) as fh:
        return list(csv.DictReader(fh))


def test_csv_without_window_columns(tmp_path):
    rows = _prepare(tmp_path, ['fast5_path', 'locus', 'read_name', 'reverse'],
                    [['a.fast5', 'LOC', 'r1', 'False'], ['a.fast5', 'LOC', 'r2', 'True']])
    assert [r['read_name'] for r in rows] == ['r1', 'r2']
    assert all(r['l_start_raw'] == '' and r['r_end_raw'] == '' for r in rows)
    assert all(r['run_id'] == 'run_0' and r['saved'] == '1' for r in rows)


def test_csv_with_some_windows_empty(tmp_path):
    rows = _prepare(tmp_path, ['fast5_path', 'locus', 'read_name', 'reverse', 'l_start_raw', 'r_end_raw'],
                    [['a.fast5', 'LOC', 'r1', 'False', '100', '900'], ['a.fast5', 'LOC', 'r2', 'True', '', '']])
    assert (rows[0]['l_start_raw'], rows[0]['r_end_raw']) == ('100', '900')
    assert (rows[1]['l_start_raw'], rows[1]['r_end_raw']) == ('', '')


@pytest.mark.parametrize('missing', ['reverse', 'read_name', 'fast5_path', 'locus'])
def test_csv_missing_a_required_column(tmp_path, missing):
    header = [c for c in ['fast5_path', 'locus', 'read_name', 'reverse'] if c != missing]
    with pytest.raises(ValueError, match='required columns'):
        _prepare(tmp_path, header, [['x'] * len(header)])
    assert not os.path.exists(str(tmp_path / 'out'))
