"""CPU: locus front-end (FASTA slices without pysam, motif -> regex)."""
import json
import os

import numpy as np
import pytest

from warpstr_b200 import locus as lc


@pytest.fixture()
def fasta(tmp_path):
    seq1 = ('ACGTTGCA' * 40)[:300]
    hd = 'AGC' * 19 + 'AACAGCCGCCAC' + 'CGC' * 7
    chr4 = 'T' * 130 + 'GATTACA' * 10 + hd + 'CCATGG' * 30
    p = tmp_path / 'ref.fa'
    with open(p, 'w') as fh:
        for name, s in (('chr1', seq1), ('chr4', chr4)):
            fh.write(f'>{name} test\n')
            for i in range(0, len(s), 60):
                fh.write(s[i:i + 60] + '\n')
    return str(p), seq1, chr4, hd


def test_fetch_and_flanks(fasta):
    path, seq1, chr4, hd = fasta
    ref = lc.FastaIndex(path)
    assert ref.fetch('chr1', 1, 10) == seq1[:10]
    assert ref.fetch('chr1', 55, 130) == seq1[54:130]
    assert ref.fetch('chr4', 290, 10**9) == chr4[289:]
    start = 130 + 70 + 1
    coord = f'chr4:{start}-{start + len(hd) - 1}'
    assert lc.get_ref_pattern(coord, ref)[0] == hd
    left, right = lc.get_flanks(coord, ref, 110, reverse=False)
    assert left == chr4[start - 1 - 110:start - 1] and right == chr4[start - 1 + len(hd):start - 1 + len(hd) + 110]
    rl, rr = lc.get_flanks(coord, ref, 110, reverse=True)
    assert rl == lc.reverse_complement(right) and rr == lc.reverse_complement(left)
    with open(path + '.fai', 'w') as fh:                        # an existing .fai is honoured
        for name, (ln, off, lb, lw) in ref.index.items():
            fh.write(f'{name}\t{ln}\t{off}\t{lb}\t{lw}\n')
    assert lc.FastaIndex(path).fetch('chr4', start, start + 5) == hd[:6]
    with pytest.raises(KeyError):
        ref.fetch('chrX', 1, 2)


def test_motif_to_regex(fasta):
    path, _, chr4, hd = fasta
    seq, note = lc.prepare_sequence(hd, 'AGC,CGC')
    assert seq == '(AGC)AACAGCCGCCAC(CGC)'
    assert note == '(AGC)[19]AACAGCCGCCAC(CGC)[7]'
    assert lc.prepare_sequence('AAATAAATAAATGAAAT', 'AAAT')[0] == '(AAAT)GAAAT'
    start = 130 + 70 + 1
    got, _ = lc.locus_sequence(f'chr4:{start}-{start + len(hd) - 1}', 'AGC,CGC', None, path)
    assert got == '(AGC)AACAGCCGCCAC(CGC)'
    assert lc.locus_sequence('x', None, '(cag)', path)[0] == '(CAG)'
    assert lc.process_coord('chr4:3,074,878-3,074,967') == ('chr4', 3074878, 3074967)
    with pytest.raises(ValueError):
        lc.prepare_sequence('A', 'AGC')


def test_motif_walk_equals_reference():
    """What Locus.prepare_sequence of the reference returned for these sequences and motifs (stored in
    golden/reference_pin.npz, see tests/test_reference_pin.py)."""
    z = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_pin.npz'))
    cases = json.loads(str(z['cases']))['motif_walk']
    assert len(cases) == 5
    for seq, motif, want in cases:
        assert list(lc.prepare_sequence(seq, motif)) == want, (seq, motif)
