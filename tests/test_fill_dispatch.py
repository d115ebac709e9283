"""CPU: every specialised DP-fill kernel instantiation has a target automaton that plans onto it.

dtw.cu compiles ``dtw_fill_kernel`` for each (chain slots, generic slots, candidate encoding, dwell)
its WSTR_CASE lines and launch_fill_deg reach; api.cu's build_layout chooses among the same splits
(kSplits).  tests/test_gpu_layouts.py runs every one of them against the oracle; this file checks,
without a GPU, that the two tables agree and that the targets reach exactly the instantiations."""
import numpy as np
import pytest

import _layouts as lay


def test_splits_match_the_fill_cases():
    """A split build_layout may choose without a WSTR_CASE would fail only at launch time
    (WSTR_ERR_UNSUPPORTED); a WSTR_CASE without a split is never run."""
    assert lay.split_cases() == lay.fill_cases()


def test_instantiation_table():
    cases = lay.INSTANTIATIONS
    assert len(cases) == len(set(cases)) == 65
    assert len(lay.fill_cases()) == 22
    # every split at the default dwell has the low layouts once it has two generic slots, the graded one
    # from three; the other dwells only the uniform ones
    for kc, kg, deg, mv in cases:
        assert deg in (2, 4) or (mv == 4 and kg >= (3 if deg == 242 else 2))
    modes = {c: lay.store_mode(c) for c in cases}
    assert set(modes.values()) == {'aligned', 'rpw1', 'shift'}
    assert any(m == 'rpw1' and c[3] == 4 for c, m in modes.items())


def test_every_instantiation_has_one_target():
    assert set(lay.REGEX) | set(lay.LADDER) == set(lay.INSTANTIATIONS)
    assert not set(lay.REGEX) & set(lay.LADDER)


@pytest.mark.parametrize('case', lay.INSTANTIATIONS, ids=lay.case_id)
def test_target_plans_onto_its_instantiation(built_lib, case):
    from warpstr_b200 import _lib
    t = lay.get(case)
    a = t.automaton()
    kc, kg, deg, mv = case
    info, sop = _lib.automaton_plan(a.in_ptr, a.in_idx, a.n_states, mv)
    assert (info['chain_slots'], info['generic_slots'], info['unrolled_in_degree']) == (kc, kg, deg)
    lay.assert_layout_invariants(a.in_ptr, a.in_idx, a.n_states, info, sop, case)
    # the quantised form has the same graph, so the same plan
    q = t.automaton(quantised=True)
    assert np.array_equal(q.in_ptr, a.in_ptr) and np.all(q.values * 8 == np.round(q.values * 8))
    # the end band: closed at the target's flank, open at flank_open where the graph has a back edge
    assert a.band_closed(t.flank)
    assert t.flank_open is not None and not a.band_closed(t.flank_open)
    assert a.endstate == a.n_states - 1 and np.all(np.diff(a.seq_idx) >= 0)


def test_targets_cover_the_instantiations(built_lib):
    """The union of the targets' plans is the instantiation table: a new WSTR_CASE without a target
    fails here."""
    from warpstr_b200 import _lib
    planned = set()
    for case in lay.INSTANTIATIONS:
        a = lay.get(case).automaton()
        info, _ = _lib.automaton_plan(a.in_ptr, a.in_idx, a.n_states, case[3])
        planned.add((info['chain_slots'], info['generic_slots'], info['unrolled_in_degree'], case[3]))
    assert planned == set(lay.INSTANTIATIONS)
    print(f'{len(planned)} of {len(lay.INSTANTIATIONS)} instantiations targeted; kSplits in sync with dtw.cu')


@pytest.mark.parametrize('case', [(6, 4, 2, 4), (12, 4, 242, 4), (6, 2, 2, 8)], ids=lay.case_id)
def test_reads_hold_every_state_mv_samples(case):
    """The read generator: 1 500-6 000 samples, dwell >= mv, quantised reads on the 1/8 grid."""
    t = lay.get(case)
    for quantised in (False, True):
        for x in t.reads(3, seed=1, quantised=quantised):
            assert 1500 <= len(x) <= 6000, len(x)
            if quantised:
                assert np.all(x * 8 == np.round(x * 8))
