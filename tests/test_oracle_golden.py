"""CPU: the oracle (numpy + C restatements) reproduces every golden vector that
oracle/make_golden.py took from the unmodified reference."""
import json
import os

import numpy as np
import pytest

from oracle import caller_oracle as co
from oracle import normalize_oracle as no
from warpstr_b200.automata import StateAutomata
from warpstr_b200.pore_model import get_pore_model

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(scope='module')
def caller_gold():
    z = np.load(os.path.join(GOLD, 'caller.npz'))
    return z, json.loads(str(z['cases']))


def _tables(case):
    sta = StateAutomata(case['reverse_regex'] if case['reverse'] else case['template_regex'])
    return co.tables_from(sta)


@pytest.mark.parametrize('impl', ['rows', 'c'])
def test_caller_oracle_matches_reference_goldens(caller_gold, oracle_c, impl):
    z, cases = caller_gold
    for case in cases:
        k = case['key']
        tb = _tables(case)
        got = co.run_read(z[f'{k}_signal'], tb, case['flank'], case['reverse'], impl=impl)
        assert np.array_equal(got.trace1, z[f'{k}_ref_trace1']), k
        assert np.array_equal(got.rescaled, z[f'{k}_ref_rescaled']), k
        T = len(got.trace1)
        assert np.array_equal(got.badmask, np.unpackbits(z[f'{k}_ref_badmask'])[:T].astype(bool)), k
        assert np.array_equal(got.trace2, z[f'{k}_ref_trace2']), k
        assert got.seq == case['seq'] and got.resc_seq == case['resc_seq'], k
        assert got.cost == case['cost'] and got.resc_cost == case['resc_cost'], k


def test_bulk_oracle_equals_the_plain_one(caller_gold, oracle_c):
    """run_read(bulk=True) -- array slices and whole-window t statistics instead of per-sample Python
    lists, what the 10^3..10^4-read parity checks use -- gives the reference's goldens bit for bit."""
    z, cases = caller_gold
    for case in cases:
        k = case['key']
        got = co.run_read(z[f'{k}_signal'], _tables(case), case['flank'], case['reverse'], impl='c', bulk=True)
        T = len(got.trace1)
        assert np.array_equal(got.badmask, np.unpackbits(z[f'{k}_ref_badmask'])[:T].astype(bool)), k
        assert np.array_equal(got.trace2, z[f'{k}_ref_trace2']), k
        assert got.seq == case['seq'] and got.resc_seq == case['resc_seq'], k
        assert got.cost == case['cost'] and got.resc_cost == case['resc_cost'], k


@pytest.mark.parametrize('bulk', [False, True])
def test_midstage_functions_on_the_reference_traces(caller_gold, oracle_c, bulk):
    """after_first_pass / after_second_pass, fed with the reference's own traces and no DP, give the
    reference's rescaled signal, bad-repeat mask and costs; the pooled driver over them gives the same and
    the sequences (what tests/test_gpu_midstage.py holds the device's mid-stage to)."""
    from oracle import bulk as ob
    z, cases = caller_gold
    kn = co.Knobs()
    for case in cases:
        k = case['key']
        tb = _tables(case)
        x, t1, t2 = z[f'{k}_signal'], z[f'{k}_ref_trace1'], z[f'{k}_ref_trace2']
        p1 = co.after_first_pass(x, t1, tb, kn, bulk)
        assert np.array_equal(p1.rescaled, z[f'{k}_ref_rescaled']), k
        assert np.array_equal(p1.badmask, np.unpackbits(z[f'{k}_ref_badmask'])[:len(x)].astype(bool)), k
        assert p1.cost == case['cost'], k
        assert co.after_second_pass(p1.rescaled, t2, tb, kn, bulk).cost == case['resc_cost'], k
        if bulk:
            rx = case['reverse_regex'] if case['reverse'] else case['template_regex']
            g = ob.run_midstage([rx], case['flank'], [x], [t1], [t2], [0], [case['reverse']], workers=1)[0]
            assert g['status'] == 0, k
            assert np.array_equal(g['rescaled'], p1.rescaled) and np.array_equal(g['mask'], p1.badmask), k
            assert (g['seq1'], g['seq2']) == (case['seq'], case['resc_seq']), k
            assert (g['cost1'], g['cost2']) == (case['cost'], case['resc_cost']), k
            assert g['m'] > 3 and g['run_hist'].sum() == len(co.state_transitions(t1)), k


def test_fill_matrices_bit_identical(caller_gold, oracle_c):
    z, cases = caller_gold
    for case in cases[:6]:
        k = case['key']
        tb = _tables(case)
        x = z[f'{k}_signal']
        m0 = np.zeros(len(x), dtype=bool)
        D_rows, _ = co.fill_rows(x, tb, m0, 4, case['flank'])
        D_c = oracle_c.fill(x, tb, m0, 4, case['flank'])
        assert np.array_equal(D_rows[::97], z[f'{k}_ref_D1_rows']), k
        assert np.array_equal(D_c[::97], z[f'{k}_ref_D1_rows']), k
        assert np.array_equal(D_c[-1], z[f'{k}_ref_D1_last']), k


def test_scalar_port_small_case(caller_gold):
    """The cell-by-cell port (the timed CPU baseline) on the shortest golden read."""
    z, cases = caller_gold
    case = [c for c in cases if c['key'] == 'AAAT_F40_1'][0]
    tb = _tables(case)
    got = co.run_read(z['AAAT_F40_1_signal'], tb, case['flank'], case['reverse'], impl='scalar')
    assert np.array_equal(got.trace1, z['AAAT_F40_1_ref_trace1'])
    assert got.resc_seq == case['resc_seq'] and got.resc_cost == case['resc_cost']


def test_backtrack_closest_equals_pointer_following(caller_gold):
    z, cases = caller_gold
    case = cases[0]
    tb = _tables(case)
    x = z[f"{case['key']}_signal"]
    m0 = np.zeros(len(x), dtype=bool)
    D, ptr = co.fill_rows(x, tb, m0, 4, case['flank'])
    assert np.array_equal(co.backtrack_closest(D, x, tb, m0, 4), co.backtrack_ptr(ptr, tb, m0, 4))


def test_normalize_oracle_matches_goldens():
    z = np.load(os.path.join(GOLD, 'normalize.npz'))
    for case in json.loads(str(z['cases'])):
        k = case['key']
        raw = z[f'{k}_raw']
        assert np.array_equal(no.brute_remove(raw), z[f'{k}_ref_brute']), k
        with np.errstate(all='ignore'):
            got = no.get_data_processed(raw, (case['lo'], case['hi']), 'Brute')
            assert np.array_equal(got, z[f'{k}_ref_norm_brute'], equal_nan=True), k
            got = no.get_data_processed(raw, (case['lo'], case['hi']), 'None')
            assert np.array_equal(got, z[f'{k}_ref_norm_none'], equal_nan=True), k
        if f'{k}_ref_norm_median3' in z:
            for mode in ('median3', 'median5'):
                got = no.get_data_processed(raw, (case['lo'], case['hi']), mode)
                assert np.array_equal(got, z[f'{k}_ref_norm_{mode}']), (k, mode)


def test_pore_model_matches_goldens():
    z = np.load(os.path.join(GOLD, 'pore_model.npz'))
    pm = get_pore_model()
    assert pm.kmersize == 6
    assert list(z['kmers']) == pm.kmers
    assert np.array_equal(pm.level_norm, z['ref_level_norm'])
    sq = np.load(os.path.join(GOLD, 'squiggle.npz'))
    seq = str(sq['seq'])
    got = pm.get_values([seq[i:i + 6] for i in range(len(seq) - 5)])
    assert np.array_equal(got, sq['ref_signal'])
    with pytest.raises(IndexError):
        pm.get_value('ACGTNA')
