"""CPU: the oracle and the product's host code against what the UNMODIFIED reference returned on
the same inputs.  The reference's answers are stored in golden/reference_pin.npz: they were recorded
from this code at the commit where every one of these comparisons last passed against the live
reference (af33a0e), so that the pins hold on any machine, without the reference."""
import hashlib
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


@pytest.fixture(scope='module')
def pin():
    z = np.load(os.path.join(GOLD, 'reference_pin.npz'))
    return json.loads(str(z['cases'])), z


def test_automaton_builder_against_reference(pin):
    from warpstr_b200.automata import StateAutomata
    cases, _ = pin
    assert len(cases['automata']) == 6
    for want in cases['automata']:
        b = StateAutomata(want['seq'])
        assert want['kmers'] == b.kmers
        assert want['values'] == list(b.values)
        assert want['incoming'] == [list(b.incoming_of(i)) for i in range(b.n_states)]
        assert want['mask'] == b.mask and want['endstate'] == b.endstate


def test_oracle_against_reference_run(pin):
    from oracle import caller_oracle as co
    from warpstr_b200.automata import StateAutomata
    cases, z = pin
    want = cases['run']
    x = z['run_signal']
    tb = co.tables_from(StateAutomata(want['regex']))
    got = co.run_read(x, tb, want['flank'], want['reverse'], impl='c')
    assert (got.seq, got.resc_seq, got.cost, got.resc_cost) == (want['seq'], want['resc_seq'], want['cost'], want['resc_cost'])
    D = co.fill_scalar(x, tb, np.full(len(x), False), 4, want['flank'])
    assert list(D.shape) == want['fill_shape']
    assert hashlib.sha256(np.ascontiguousarray(D, dtype=np.float64).tobytes()).hexdigest() == want['fill_sha256']


def test_wrapper_helpers_against_reference(pin):
    from warpstr_b200.wrapper import CallerWrapper
    want = pin[0]['wrapper']
    mine = CallerWrapper.__new__(CallerWrapper)
    for pat, w in want['units'].items():
        assert json.loads(json.dumps(mine.break_into_units(pat))) == w['break_into_units']
        assert mine.reverse_uniq_sequence(pat) == w['reverse_uniq_sequence']
    mine.units, mine.repeat_units, mine.offsets = mine.break_into_units('((CAGG){CAGM})(CAGA)(CA)')
    assert len(want['collapse']) == 4
    for seq, w in want['collapse'].items():
        assert json.loads(json.dumps(mine.collapse_repeats(seq))) == w


def test_normalize_oracle_against_reference(pin):
    from oracle import normalize_oracle as no
    z = pin[1]
    raw = z['norm_raw']
    assert np.array_equal(raw, np.random.default_rng(5).integers(200, 1100, size=5001).astype(np.int16))
    assert np.array_equal(no.brute_remove(raw), z['norm_brute_remove'])
    assert np.array_equal(no.normalize_signal_mad(raw), z['norm_mad'])


def test_bundled_reads_against_reference_run():
    """Two of the reference's own bundled test reads (real nanopore signal, golden/c1_bundled.npz):
    the oracle's normalisation and call against what the fixture holds -- the answers the unmodified
    reference's normalisation and WarpSTR.run gave for these reads, and what the GPU path is compared
    with in tests/test_gpu_c1.py."""
    from oracle import caller_oracle as co
    from oracle import normalize_oracle as no
    from warpstr_b200 import templates as tmpl
    from warpstr_b200.automata import StateAutomata
    z = np.load(os.path.join(GOLD, 'c1_bundled.npz'))
    left, right, seq, F = str(z['left']), str(z['right']), str(z['sequence']), int(z['flank_length'])
    regex = {False: left + seq + right,
             True: tmpl.reverse_complement(right) + tmpl.reverse_uniq_sequence(seq) + tmpl.reverse_complement(left)}
    order = np.argsort(z['r_end_raw'] - z['l_start_raw'])[:2]            # the two shortest windows
    for i in order:
        raw = np.cumsum(z[f'raw_delta{i}'].astype(np.int64)).astype(np.int16)
        norm = no.normalize_signal_mad(no.brute_remove(raw))              # Fast5.get_data_processed, fast5.py:45-57
        x = np.ascontiguousarray(norm[int(z['l_start_raw'][i]):int(z['r_end_raw'][i]) + 1])
        rev = bool(z['reverse'][i])
        got = co.run_read(x, co.tables_from(StateAutomata(regex[rev])), F, rev, impl='c')
        assert got.seq == str(z['seq'][i]) and got.resc_seq == str(z['resc_seq'][i])
        assert got.cost == z['cost1'][i] and got.resc_cost == z['cost2'][i]
        assert len(got.resc_seq) in (40, 44)
