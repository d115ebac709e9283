"""CPU: host-side logic of the product (config, packing, the host mid-stage, kernel layout
planning, wrapper helpers)."""
import json
import os

import numpy as np
import pytest

import _layouts as lay
from warpstr_b200 import config as cfg
from warpstr_b200 import midstage, synth
from warpstr_b200.automata import StateAutomata
from warpstr_b200.caller import pack_masks, pack_signals

GOLD = os.path.join(os.path.dirname(__file__), 'golden')


def test_config_defaults_and_yaml(tmp_path):
    c = cfg.config_from_dict({'loci': [{'name': 'HD', 'coord': 'chr4:1-2', 'sequence': '(agc)AAC'}]})
    assert c.caller_config.min_values_per_state == 4 and c.caller_config.states_in_segment == 6
    assert c.rescaler_config.threshold == 0.5 and c.rescaler_config.method == 'mean'
    assert c.flank_length == 110 and c.loci[0].sequence == '(AGC)AAC'
    p = tmp_path / 'c.yaml'
    p.write_text('output: out\nreference_path: ref.fa\nflank_length: 80\n'
                 'tr_calling_config:\n  min_values_per_state: 5\nrescaling:\n  threshold: 0.4\n'
                 'loci:\n  - name: X\n    coord: chr1:5-9\n    sequence: (CAG)\n    flank_length: 60\n')
    c = cfg.load_config(str(p))
    assert c.caller_config.min_values_per_state == 5 and c.caller_config.spike_removal == 'Brute'
    assert c.rescaler_config.threshold == 0.4 and c.rescaler_config.max_std == 0.5
    assert c.locus_flank_length(c.loci[0]) == 60 and c.flank_length == 80
    assert os.path.exists(c.pore_model_path)
    with pytest.raises(AssertionError):
        cfg.CallerConfig(spike_removal='median7')
    with pytest.raises(AssertionError):
        cfg.RescalerConfig(method='mode')
    (tmp_path / 'noloci.yaml').write_text('output: x\n')
    with pytest.raises(KeyError):
        cfg.load_config(str(tmp_path / 'noloci.yaml'))
    with pytest.raises(FileNotFoundError):
        cfg.load_config(str(tmp_path / 'missing.yaml'))


def test_pack_signals_alignment_and_masks():
    sigs = [np.arange(5, dtype=np.float64), np.arange(8, dtype=np.float64) + 10, np.zeros(1)]
    host, off, lengths = pack_signals(sigs)
    assert (off % 2 == 0).all() and list(lengths) == [5, 8, 1]
    buf = host.numpy()
    for s, o in zip(sigs, off):
        assert np.array_equal(buf[o:o + len(s)], s)
    assert host.numel() >= off[-1] + 2
    masks = [np.array([1, 0, 1] + [0] * 40 + [1], dtype=bool), np.zeros(3, dtype=bool), np.ones(32, dtype=bool)]
    words, moff = pack_masks(masks)
    assert list(moff) == [0, 2, 3]
    assert words[0] == 0b101 and words[1] == 1 << (43 - 32) and words[2] == 0 and words[3] == 0xffffffff


def test_host_midstage_reproduces_reference_goldens():
    z = np.load(os.path.join(GOLD, 'caller.npz'))
    cases = json.loads(str(z['cases']))
    cc, rc = cfg.CallerConfig(), cfg.RescalerConfig()
    for case in cases:
        k = case['key']
        sta = StateAutomata(case['reverse_regex'] if case['reverse'] else case['template_regex'])
        x = z[f'{k}_signal']
        t1 = z[f'{k}_ref_trace1'].astype(np.int64)
        p1 = midstage.after_pass(t1, x, sta.values, sta.rep_mask.astype(bool), cc, rc, False)
        assert np.array_equal(p1.rescaled, z[f'{k}_ref_rescaled']), k
        assert np.array_equal(p1.badmask, np.unpackbits(z[f'{k}_ref_badmask'])[:len(x)].astype(bool)), k
        assert (p1.start, p1.end) == (case['start'], case['end']) and p1.cost == case['cost'], k
        t2 = z[f'{k}_ref_trace2'].astype(np.int64)
        p2 = midstage.after_pass(t2, p1.rescaled, sta.values, sta.rep_mask.astype(bool), cc, rc, True)
        assert p2.cost == case['resc_cost'], k


def test_host_midstage_errors_carry_the_reference_exception_type():
    cc, rc = cfg.CallerConfig(), cfg.RescalerConfig()
    sta = StateAutomata('ACGTTGCATG' + '(CAG)' + 'TTGACCAGTA')
    x = np.zeros(50)
    trace = np.zeros(50, dtype=np.int64)                 # never leaves state 0: nothing to fit
    with pytest.raises(midstage.ReadError) as e:
        midstage.after_pass(trace, x, sta.values, sta.rep_mask.astype(bool), cc, rc, False)
    assert e.value.kind is TypeError                     # splrep: m > k must hold
    runs = midstage.run_lengths(trace)
    with pytest.raises(midstage.ReadError) as e:
        midstage.mask_bad_repeats(x, sta.rep_mask.astype(bool), runs, cc)
    assert e.value.kind is IndexError                    # trues[0]


def test_kernel_layout_plan_invariants(built_lib):
    from warpstr_b200 import _lib
    for name in ('AAAT', 'HD', 'FMR1', 'FMR1_MGG', 'DM2', 'CAN', 'RFC1', 'C9ORF72_100'):
        locus = synth.make_locus(name, seed=3)
        for rx in (locus.template_regex, locus.reverse_regex):
            sta = StateAutomata(rx)
            info, sop = _lib.automaton_plan(sta.in_ptr, sta.in_idx, sta.n_states)
            lay.assert_layout_invariants(sta.in_ptr, sta.in_idx, sta.n_states, info, sop, name)


def test_layout_plan_never_refuses_what_the_reference_accepts(built_lib):
    """An automaton or dwell setting without a specialised layout plans onto the catch-all kernel
    (all-zero plan), it is not an error; only what no kernel can hold is."""
    from warpstr_b200 import _lib
    S = 600                                              # more than the 512 register-resident positions
    ptr = np.arange(S + 1, dtype=np.int32)
    ptr[1:] -= 1
    ptr[0] = 0
    idx = np.arange(S - 1, dtype=np.int32)
    info, sop = _lib.automaton_plan(ptr, idx, S)
    assert info['chain_slots'] == 0 and info['generic_slots'] == 0 and len(sop) == 0
    with pytest.raises(_lib.WarpstrError):               # states x dwell beyond the shared memory of an SM
        _lib.automaton_plan(ptr, idx, S, 64)
    # every dwell setting on every locus shape of the test set plans: specialised kernels for 2..8
    # (the 324-state reverse strand of (CAN) only at the default 4), the catch-all beyond
    for name in ('HD', 'DM2', 'CAN', 'RFC1', 'FMR1_MGG'):
        locus = synth.make_locus(name, seed=3)
        for rx in (locus.template_regex, locus.reverse_regex):
            sta = StateAutomata(rx)
            for mv in (2, 3, 4, 5, 6, 7, 8, 12):
                info, _ = _lib.automaton_plan(sta.in_ptr, sta.in_idx, sta.n_states, mv)
                if mv > 8:
                    assert info['chain_slots'] == 0
                elif sta.n_states <= 320 or mv == 4:
                    assert info['chain_slots'] > 0, (name, mv, info)


def test_wrapper_unit_helpers():
    from warpstr_b200.wrapper import CallerWrapper
    w = CallerWrapper.__new__(CallerWrapper)
    units, reps, offs = w.break_into_units('((CAGG){CAGM})(CAGA)(CA)')
    assert units == ['((CAGG){CAGM})', '(CAGA)', '(CA)'] and offs == [0, 0, 0]
    assert reps == [['CAGG', 'CAGGCAGA', 'CAGGCAGC'], ['CAGA'], ['CA']]
    units, reps, offs = w.break_into_units('(AGC)AACAGCCGCCAC(CGC)')
    assert units == ['(AGC)', '(CGC)'] and offs == [0, 12]
    w.repeat_units, w.offsets = reps, offs
    assert w.collapse_repeats('AGC' * 5 + 'AACAGCCGCCAC' + 'CGC' * 3) == [[5], [3]]
    assert w.reverse_uniq_sequence('(AGC)AAC') == 'GTT(GCT)'


def test_synthetic_batch_generator_is_consistent():
    locus = synth.make_locus('HD', seed=2)
    sig, off, lengths, rev, truth = synth.make_read_batch(locus, 50, seed=9)
    assert (off % 2 == 0).all() and len(sig) >= off[-1] + lengths[-1]
    assert set(np.unique(rev)) <= {0, 1} and (truth % 3 == 0).all()
    again = synth.make_read_batch(locus, 50, seed=9)
    assert np.array_equal(sig, again[0]) and np.array_equal(lengths, again[2])
    assert (np.diff(off) >= lengths[:-1]).all()


def test_exact_division_identity_the_midstage_relies_on(tmp_path):
    """The mid-stage and the normalisation kernel divide by repeated divisors with y = RN(1/d) and two FMA
    correction steps (csrc/wstr_internal.h); oracle/div_identity.c checks on the host that this gives the bits
    of a/d (random and adversarial significands, the kernels' exponent ranges, and the normalisation's
    (sample - shift) / scale family).  Needs gcc and a CPU with FMA."""
    import os
    import shutil
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if shutil.which('gcc') is None:
        pytest.skip('no gcc')
    try:
        if ' fma ' not in open('/proc/cpuinfo').read():
            pytest.skip('host CPU has no FMA')
    except OSError:
        pytest.skip('cannot read /proc/cpuinfo')
    exe = str(tmp_path / 'div_identity')
    subprocess.check_call(['gcc', '-O2', '-mfma', '-ffp-contract=off', '-o', exe,
                           os.path.join(root, 'oracle', 'div_identity.c'), '-lm'])
    out = subprocess.run([exe, '5000000'], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert 'two_step_mismatches=0' in out.stdout


def test_pore_model_path_of_a_config(tmp_path):
    """The reference's default path resolves to the bundled table; a user's own path that does not
    exist fails like the reference (pore_model.py:22-24) instead of silently using another model."""
    from warpstr_b200 import config as cfg
    base = {'loci': [{'name': 'x', 'sequence': '(AAAT)'}], 'output': str(tmp_path)}
    c = cfg.config_from_dict(dict(base))
    assert c.pore_model_path == cfg.DEFAULT_PORE_MODEL
    c = cfg.config_from_dict(dict(base, pore_model_path='example/deps/template_median68pA.model'))
    assert c.pore_model_path == cfg.DEFAULT_PORE_MODEL
    with pytest.raises(FileNotFoundError):
        cfg.config_from_dict(dict(base, pore_model_path=str(tmp_path / 'r10_custom.model')))
    own = tmp_path / 'own.model'
    own.write_text(open(cfg.DEFAULT_PORE_MODEL).read())
    assert cfg.config_from_dict(dict(base, pore_model_path=str(own))).pore_model_path == str(own)


def test_product_package_does_not_import_scipy_or_the_oracle():
    """scipy is the host evaluation's dependency for flagged reads only; the oracle is test infrastructure."""
    import subprocess
    import sys
    code = ("import sys; import warpstr_b200.caller, warpstr_b200.wrapper, warpstr_b200.shard, warpstr_b200.normalize; "
            "print(sorted(m for m in sys.modules if m.split('.')[0] in ('scipy', 'oracle')))")
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert out.returncode == 0 and out.stdout.strip() == '[]', out.stdout + out.stderr
