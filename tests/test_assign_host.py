"""CPU: the host side of the flank assignment (DESIGN.md section 4.6): the decision rule, the flank chains, the
overview writer shared with caller_only.prepare, the command line, and the rule's margin on the C oracle."""
import csv
import os

import numpy as np
import pytest

from warpstr_b200 import assign, synth
from warpstr_b200.wrapper import flanks_from_template

F, NF, NP = 0, 1, 2      # LOCATE_FOUND, LOCATE_NOT_FOUND, LOCATE_NO_PATH


def _table(entries, n_reads=1, n_loci=1):
    """{(read, locus, chain): (lo, hi, score, status)} -> the four [n_reads, 4 * n_loci] arrays; absent entries
    are NOT_FOUND."""
    lo = np.full((n_reads, 4 * n_loci), -1, np.int32)
    hi = lo.copy()
    score = np.full((n_reads, 4 * n_loci), 50.0)
    status = np.full((n_reads, 4 * n_loci), NF, np.int32)
    for (r, k, c), (a, b, s, st) in entries.items():
        lo[r, 4 * k + c], hi[r, 4 * k + c], score[r, 4 * k + c], status[r, 4 * k + c] = a, b, s, st
    return lo, hi, score, status


def _hits(res):
    return list(zip(res['read'].tolist(), res['locus'].tolist(), res['strand'].tolist()))


def test_one_strand_passing():
    t = _table({(0, 0, 0): (100, 600, -90.0, F), (0, 0, 1): (900, 1400, -80.0, F)})
    res = assign.choose_loci(*t)
    assert _hits(res) == [(0, 0, 0)]
    assert (res['left_lo'][0], res['left_hi'][0], res['right_lo'][0], res['right_hi'][0]) == (100, 600, 900, 1400)
    assert (res['left_score'][0], res['right_score'][0]) == (-90.0, -80.0)
    t = _table({(0, 0, 2): (100, 600, -10.0, F), (0, 0, 3): (900, 1400, -5.0, F), (0, 0, 0): (1, 2, -500.0, F)})
    assert _hits(assign.choose_loci(*t)) == [(0, 0, 1)]


def test_both_strands_lower_sum_wins_and_a_tie_goes_to_the_template():
    both = {(0, 0, 0): (10, 20, -50.0, F), (0, 0, 1): (30, 40, -50.0, F),
            (0, 0, 2): (10, 20, -70.0, F), (0, 0, 3): (30, 40, -31.0, F)}
    res = assign.choose_loci(*_table(both))
    assert _hits(res) == [(0, 0, 1)] and res['left_score'][0] == -70.0
    both[(0, 0, 3)] = (30, 40, -30.0, F)          # -100 either way: the template
    assert _hits(assign.choose_loci(*_table(both))) == [(0, 0, 0)]
    # a tie in the sums, not in the parts
    both[(0, 0, 2)], both[(0, 0, 3)] = (10, 20, -99.5, F), (30, 40, -0.5, F)
    assert _hits(assign.choose_loci(*_table(both))) == [(0, 0, 0)]


def test_flanks_out_of_order_or_touching_do_not_pass():
    for lo2 in (20, 15, 5):      # right.lo == left.hi, inside, before
        t = _table({(0, 0, 0): (10, 20, -50.0, F), (0, 0, 1): (lo2, lo2 + 10, -50.0, F)})
        assert _hits(assign.choose_loci(*t)) == []
    t = _table({(0, 0, 0): (10, 20, -50.0, F), (0, 0, 1): (21, 30, -50.0, F)})
    assert _hits(assign.choose_loci(*t)) == [(0, 0, 0)]


@pytest.mark.parametrize('missing', [NP, NF])
def test_a_flank_without_a_path_or_not_found(missing):
    t = _table({(0, 0, 0): (-1, -1, np.inf, missing) if missing == NP else (10, 20, 3.0, NF),
                (0, 0, 1): (30, 40, -50.0, F), (0, 0, 2): (10, 20, -1.0, F), (0, 0, 3): (5, 8, -1.0, F)})
    assert _hits(assign.choose_loci(*t)) == []


def test_a_read_passing_two_loci_is_assigned_to_both():
    t = _table({(1, 0, 0): (10, 20, -50.0, F), (1, 0, 1): (30, 40, -50.0, F),
                (1, 2, 2): (10, 20, -50.0, F), (1, 2, 3): (30, 40, -50.0, F),
                (0, 1, 0): (10, 20, -50.0, F), (0, 1, 1): (30, 40, -50.0, F)}, n_reads=2, n_loci=3)
    assert _hits(assign.choose_loci(*t)) == [(0, 1, 0), (1, 0, 0), (1, 2, 1)]


def test_no_reads():
    res = assign.choose_loci(*(a[:0] for a in _table({}, n_loci=2)))
    assert all(len(v) == 0 for v in res.values()) and set(res) == set(assign.HIT_FIELDS)


def test_panel_chains():
    loci = [synth.make_locus(n, seed=5 + k) for k, n in enumerate(('HD', 'CAN'))]
    p = assign.Panel([(L.name, flanks_from_template(L.left, L.right)) for L in loci])
    assert p.names == ['HD', 'CAN'] and len(p.chains) == 8
    for c in p.chains:          # a 110-base flank: a chain of 105 6-mer states, the end state last
        assert c.n_states == 105 and c.endstate == 104 and list(c.in_ptr) == [0] + list(range(105))
        assert list(c.in_idx) == list(range(104))
    f = flanks_from_template(loci[1].left, loci[1].right)
    assert p.chains[4].kmers[0] == f.template.left[:6] and p.chains[7].kmers[-1] == f.reverse.right[-6:]


def test_panel_from_config_reads_the_locus_flanks(tmp_path):
    from warpstr_b200.config import Config, LocusConfig
    L = synth.make_locus('HD', seed=9)
    _write_flanks(str(tmp_path / 'HD'), L.left, L.right)
    cfg = Config(output=str(tmp_path), loci=[LocusConfig(name='HD', sequence=L.sequence)])
    p = assign.Panel.from_config(cfg)
    assert p.names == ['HD'] and p.chains[0].sequence == L.left and p.chains[1].sequence == L.right


def _write_flanks(path, left, right):
    from warpstr_b200 import templates as tmpl
    f = flanks_from_template(left, right)
    os.makedirs(os.path.join(path, tmpl.LOCUS_INFO_SUBDIR), exist_ok=True)
    with open(os.path.join(path, tmpl.LOCUS_INFO_SUBDIR, tmpl.LOCUS_FLANKS), 'w') as fh:
        fh.write('type,sequence\n')
        for k, v in (('left_flank_template', f.template.left), ('right_flank_template', f.template.right),
                     ('left_flank_reverse', f.reverse.left), ('right_flank_reverse', f.reverse.right)):
            fh.write(f'{k},{v}\n')


def test_overview_writer(tmp_path):
    from warpstr_b200.caller_only import write_overviews
    rows = {'A': [['x.pod5', 'A', 'r1', 'True', '', '', 'run_0', '1']], 'B': [['y,z.fast5', 'B', 'r2', 'False', '', '',
                                                                             'run_0', '1']]}
    written = write_overviews(str(tmp_path), assign.OVERVIEW_HEADER, rows)
    assert set(written) == {'A', 'B'}
    with open(written['B'], newline='') as fh:
        got = list(csv.reader(fh))
    assert got == [assign.OVERVIEW_HEADER] + rows['B']
    with open(written['A'], 'rb') as fh:
        assert fh.read() == (','.join(assign.OVERVIEW_HEADER) + '\r\nx.pod5,A,r1,True,,,run_0,1\r\n').encode()


def test_scan_runs(tmp_path):
    for p in ('b/2.pod5', 'b/1.FAST5', 'a/x.fast5', 'a/notes.txt', 'c.pod5'):
        os.makedirs(os.path.dirname(str(tmp_path / p)), exist_ok=True)
        (tmp_path / p).write_bytes(b'')
    got = assign.scan_runs([str(tmp_path), str(tmp_path / 'c.pod5')])
    assert [os.path.relpath(g, str(tmp_path)) for g in got] == ['c.pod5', 'a/x.fast5', 'b/1.FAST5', 'b/2.pod5']
    assert assign.scan_runs([str(tmp_path / 'a' / 'notes.txt')]) == [str(tmp_path / 'a' / 'notes.txt')]
    with pytest.raises(FileNotFoundError):
        assign.scan_runs([str(tmp_path / 'nope')])


def test_command_line(tmp_path, monkeypatch):
    cfg = tmp_path / 'cfg.yaml'
    cfg.write_text(f'output: {tmp_path / "out"}\nloci:\n  - name: HD\n    sequence: (CAG)\n')
    run = tmp_path / 'run'
    run.mkdir()
    (run / 'r.pod5').write_bytes(b'')
    seen = {}
    monkeypatch.setattr(assign, 'assign_files', lambda config, files: seen.update(config=config, files=files))
    assign.main(['--config', str(cfg), str(run)])
    assert seen['files'] == [str(run / 'r.pod5')] and [l.name for l in seen['config'].loci] == ['HD']
    with pytest.raises(SystemExit):
        assign.main(['--config', str(cfg)])           # no RUN
    with pytest.raises(SystemExit):
        assign.main([str(run)])                        # no --config
    (run / 'r.pod5').unlink()
    with pytest.raises(FileNotFoundError, match='no .fast5 or .pod5'):
        assign.main(['--config', str(cfg), str(run)])


def test_flank_rule_margin_on_the_oracle():
    """The rule on wso_locate: flanks of reads of a locus score far below zero, flank chains searched in random
    sequence (or in another locus's reads) never reach zero, at the offset 0.35 the caller uses."""
    from oracle import locate as lo_oracle
    pm = synth.get_pore_model()
    loci = [synth.make_locus(n, seed=20 + k) for k, n in enumerate(('HD', 'DM2'))]
    p = assign.Panel([(L.name, flanks_from_template(L.left, L.right)) for L in loci])
    rng = np.random.default_rng(21)
    sigs, truth = [], []
    for k, L in enumerate(loci):
        for r in synth.make_reads(L, 3, seed=22 + k):
            fill = [synth.squiggle(rng, synth.random_flank(rng, 300), pm) for _ in range(2)]
            sigs.append(np.concatenate((fill[0], r.signal, fill[1])))
            truth.append((k, int(r.reverse)))
    for _ in range(4):
        sigs.append(synth.squiggle(rng, synth.random_flank(rng, 2500), pm))
        truth.append(None)
    n, A = len(sigs), len(p.chains)
    lo, hi, score, status = lo_oracle.locate_batch([s for s in sigs for _ in range(A)], p.chains * n, 4,
                                                   threads=os.cpu_count() or 4)
    score = score.reshape(n, A)
    res = assign.choose_loci(lo.reshape(n, A), hi.reshape(n, A), score, status.reshape(n, A))
    assert _hits(res) == [(r, k, s) for r, t in enumerate(truth) if t is not None for k, s in [t]]
    for r, t in enumerate(truth):
        own = set() if t is None else {4 * t[0] + 2 * t[1], 4 * t[0] + 2 * t[1] + 1}
        for a in range(A):
            assert (score[r, a] < -150) if a in own else (score[r, a] > 0), (r, a, score[r, a])
