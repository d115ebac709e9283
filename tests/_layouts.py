"""One target automaton for every specialised DP-fill kernel instantiation (csrc/dtw.cu).

``dtw_fill_kernel<KC, KG, DEG, MV, MASKED>`` is compiled for every ``(KC, KG, DEG, MV)`` that
``launch_fill_deg`` can reach from the ``WSTR_CASE(kc, kg, mv)`` lines of dtw.cu, and which one a
locus runs on depends only on the shape of its automaton (``build_layout`` in csrc/api.cu picks the
cheapest split that fits).  ``INSTANTIATIONS`` is that set, read from the sources; ``TARGETS`` maps
each tuple to an automaton that plans onto it:

* a regex locus (``synth.SynthLocus``) where one reaches the tuple: a realistic automaton, whose reads
  are made the way ``synth.make_reads`` makes them;
* otherwise a constructed graph: a left chain, a "ladder" of positions two states wide (each state
  fed by both states of the position before), a back edge from the last ladder position to the first
  and a right chain; optionally a few four-wide positions (their successors have four incoming edges)
  and a "comb" of single-predecessor states (a spine whose states each feed one dead-end state).

Every target also comes in a quantised form: levels and samples on a 1/8 grid, so that every sum is
exact and equal candidates really tie (strict '<', list order).
"""
import os
import re
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from oracle import caller_oracle as co
from warpstr_b200 import synth
from warpstr_b200.automata import StateAutomata
from warpstr_b200.pore_model import get_pore_model
from warpstr_b200.templates import reverse_complement

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'warpstr_b200', 'csrc')
NOISE = 0.15
QUANTUM = 0.125


# ---------------------------------------------------------------------------------------------------
# the instantiation table
# ---------------------------------------------------------------------------------------------------
def fill_cases() -> set:
    """(kc, kg, mv) of every WSTR_CASE line of dtw.cu."""
    text = open(os.path.join(CSRC, 'dtw.cu')).read()
    return {tuple(int(a) for a in m) for m in re.findall(r'^\s*WSTR_CASE\((\d+),\s*(\d+),\s*(\d+)\)', text, re.M)}


def split_cases() -> set:
    """(kc, kg, mv) of every split of api.cu's kSplits (bit mv of mv_mask set = built for that dwell)."""
    text = open(os.path.join(CSRC, 'api.cu')).read()
    body = re.search(r'kSplits\[\]\s*=\s*\{(.*?)\};', text, re.S).group(1)
    out = set()
    for kc, kg, mask in re.findall(r'\{\s*(\d+),\s*(\d+),\s*(0x[0-9a-fA-F]+|\d+)\s*\}', body):
        m = int(mask, 0)
        out |= {(int(kc), int(kg), mv) for mv in range(32) if (m >> mv) & 1}
    return out


def degs(kg: int, mv: int) -> Tuple[int, ...]:
    """Candidate encodings dtw.cu's launch_fill_deg instantiates for a (kc, kg, mv) case: 2 and 4 always,
    the "low" 102 / 104 when kg >= 2 and mv == 4, the "graded" 242 when kg >= 3 and mv == 4."""
    out = (2, 4)
    if kg >= 2 and mv == 4:
        out += (102, 104)
    if kg >= 3 and mv == 4:
        out += (242,)
    return out


INSTANTIATIONS: List[Tuple[int, int, int, int]] = sorted(
    (kc, kg, d, mv) for kc, kg, mv in fill_cases() for d in degs(kg, mv))


def dir_bits(kc: int, kg: int, deg: int) -> int:
    """Direction-code bits per lane and row (dtw.cu: DirFmt<KC, KG, DEG>::NB)."""
    if deg >= 200:
        return kc + (kg - 2) + (deg - 200) % 10 + (deg - 200) // 10
    if deg >= 100:
        return kc + (kg - 1) + (deg - 100)
    return kc + kg * deg


def rows_per_word(case) -> int:
    kc, kg, deg, _ = case
    return 32 // dir_bits(kc, kg, deg)


def store_mode(case) -> str:
    """How dp_segment stores the direction words of the case: 'aligned' (RPW == mv-1, one word per
    row cycle), 'rpw1' (one row per word) or 'shift' (general shift-and-flush)."""
    rpw, mv = rows_per_word(case), case[3]
    if rpw == 1:
        return 'rpw1'
    return 'aligned' if rpw == mv - 1 else 'shift'


# ---------------------------------------------------------------------------------------------------
# automata
# ---------------------------------------------------------------------------------------------------
@dataclass
class Automaton:
    """The arrays CallerEngine.add_automaton takes."""
    values: np.ndarray
    seq_idx: np.ndarray
    in_ptr: np.ndarray
    in_idx: np.ndarray
    rep_mask: np.ndarray
    last_base: np.ndarray
    endstate: int

    @property
    def n_states(self) -> int:
        return len(self.values)

    def quantised(self) -> 'Automaton':
        return Automaton(np.round(self.values / QUANTUM) * QUANTUM, self.seq_idx, self.in_ptr, self.in_idx,
                         self.rep_mask, self.last_base, self.endstate)

    def tables(self) -> co.Tables:
        return co.Tables(values=self.values, seq_idx=self.seq_idx, in_ptr=self.in_ptr, in_idx=self.in_idx,
                         rep_mask=self.rep_mask.astype(bool), last_base=bytes(self.last_base).decode('ascii'),
                         endstate=self.endstate)

    def band_closed(self, flank: int) -> bool:
        """api.cu: no state the end band skips has an incoming edge from one it keeps."""
        after = int(self.seq_idx[-1]) - (flank - 10)
        for j in np.flatnonzero(self.seq_idx < after):
            if (self.seq_idx[self.in_idx[self.in_ptr[j]:self.in_ptr[j + 1]]] >= after).any():
                return False
        return True


def _from_preds(preds, seq_idx, rep, rng) -> Automaton:
    S = len(preds)
    ip = np.zeros(S + 1, dtype=np.int32)
    ip[1:] = np.cumsum([len(p) for p in preds])
    table = get_pore_model().table
    levels = table[np.isfinite(table)]
    seq_idx = np.asarray(seq_idx, dtype=np.int32)
    return Automaton(values=rng.choice(levels, S), seq_idx=seq_idx,
                     in_ptr=ip, in_idx=np.array([q for p in preds for q in p], dtype=np.int32),
                     rep_mask=np.asarray(rep, dtype=np.uint8),
                     last_base=np.frombuffer(b'ACGT', dtype=np.uint8)[seq_idx % 4].copy(), endstate=S - 1)


def ladder(flank: int, positions: int, merges: int = 0, comb: int = 0, seed: int = 0) -> Automaton:
    """Left chain of ``flank`` states, ``comb`` spine states with a dead-end tooth each, ``positions`` ladder
    positions (two states each, four at positions 2, 6, 10, ... for the first ``merges``), a back edge from
    the last ladder position to the first, and a right chain of ``flank`` states."""
    preds, seq, rep = [], [], []

    def add(p, s, r):
        preds.append(list(p))
        seq.append(s)
        rep.append(r)
        return len(preds) - 1

    prev = [add([], 0, False)]
    for j in range(1, flank):
        prev = [add(prev, j, False)]
    at = flank
    for _ in range(comb):
        spine = add(prev, at, True)
        add([spine], at + 1, True)
        prev = [spine]
        at += 1
    width = [2] * positions
    for m in range(merges):
        width[2 + 4 * m] = 4
    first = None
    for k in range(positions):
        cur = [add(prev, at, True) for _ in range(width[k])]
        first = cur if first is None else first
        prev = cur
        at += 1
    preds[first[0]].append(prev[0])
    for j in range(flank):
        prev = [add(prev, at + j, False)]
    return _from_preds(preds, seq, rep, np.random.default_rng([seed, flank, positions, merges, comb]))


def _regex_automaton(sta: StateAutomata) -> Automaton:
    return Automaton(values=np.asarray(sta.values, dtype=np.float64), seq_idx=np.asarray(sta.seq_idx, dtype=np.int32),
                     in_ptr=np.asarray(sta.in_ptr, dtype=np.int32), in_idx=np.asarray(sta.in_idx, dtype=np.int32),
                     rep_mask=np.asarray(sta.rep_mask, dtype=np.uint8),
                     last_base=np.asarray(sta.last_base, dtype=np.uint8), endstate=int(sta.endstate))


# ---------------------------------------------------------------------------------------------------
# targets
# ---------------------------------------------------------------------------------------------------
# (recipe, flank length, reverse strand) of a regex locus that plans onto the tuple (make_locus seed 3)
REGEX = {
    (4, 4, 104, 4): ('CAN', 80, False),
    (4, 4, 242, 4): ('CAN', 80, True),
    (6, 2, 2, 2): ('AAAT', 110, False),
    (6, 2, 2, 3): ('AAAT', 110, False),
    (6, 2, 2, 5): ('AAAT', 110, False),
    (6, 2, 2, 6): ('AAAT', 110, False),
    (6, 2, 2, 7): ('AAAT', 110, False),
    (6, 2, 2, 8): ('AAAT', 110, False),
    (6, 2, 4, 2): ('FMR1', 110, True),
    (6, 2, 4, 3): ('FMR1', 110, True),
    (6, 2, 4, 5): ('FMR1', 110, True),
    (6, 2, 4, 6): ('FMR1', 110, True),
    (6, 2, 4, 7): ('FMR1', 110, True),
    (6, 2, 4, 8): ('FMR1', 110, True),
    (6, 2, 102, 4): ('FMR1_MGG', 110, False),
    (6, 2, 104, 4): ('FMR1', 110, True),
    (6, 4, 2, 2): ('RFC1', 110, False),
    (6, 4, 2, 3): ('RFC1', 110, False),
    (6, 4, 2, 5): ('RFC1', 110, False),
    (6, 4, 2, 6): ('RFC1', 110, False),
    (6, 4, 2, 7): ('RFC1', 110, False),
    (6, 4, 2, 8): ('RFC1', 110, False),
    (6, 4, 4, 2): ('DM2', 110, False),
    (6, 4, 4, 3): ('DM2', 110, False),
    (6, 4, 4, 5): ('DM2', 110, False),
    (6, 4, 4, 6): ('DM2', 110, False),
    (6, 4, 4, 7): ('DM2', 110, False),
    (6, 4, 4, 8): ('DM2', 110, False),
    (6, 4, 102, 4): ('RFC1', 130, False),
    (6, 4, 104, 4): ('CAN', 110, False),
    (6, 4, 242, 4): ('CAN', 100, True),
    (7, 1, 2, 4): ('AAAT', 110, False),
    (7, 1, 4, 4): ('FMR1', 40, False),
    (7, 2, 102, 4): ('RFC1', 110, False),
    (7, 2, 104, 4): ('DM2', 110, False),
    (7, 4, 102, 4): ('RFC1', 140, False),
    (7, 4, 104, 4): ('CAN', 120, False),
    (7, 4, 242, 4): ('CAN', 110, True),
    (8, 1, 2, 4): ('AAAT', 130, False),
    (8, 2, 102, 4): ('HD', 140, False),
    (8, 2, 104, 4): ('DM2', 130, False),
    (8, 4, 102, 4): ('RFC1', 160, True),
    (8, 4, 104, 4): ('CAN', 130, False),
    (8, 4, 242, 4): ('CAN', 130, True),
    (12, 4, 102, 4): ('RFC1', 170, False),
    (12, 4, 104, 4): ('CAN', 150, False),
    (12, 4, 242, 4): ('CAN', 150, True),
}
# (flank, ladder positions, four-wide positions, comb length) of a constructed graph, for the tuples no
# regex locus reaches: no loop-and-flank regex has more than 32 states with two incoming edges outside
# the (6, 4) split, or a layout with two or more generic slots and states of four incoming edges that is
# neither "low" nor "graded"
LADDER = {
    (4, 4, 2, 4): (80, 40, 0, 0),
    (4, 4, 4, 4): (90, 35, 3, 0),
    (4, 4, 102, 4): (90, 12, 0, 20),
    (6, 2, 2, 4): (100, 20, 0, 0),
    (6, 2, 4, 4): (100, 20, 3, 0),
    (6, 4, 2, 4): (110, 40, 0, 0),
    (6, 4, 4, 4): (110, 40, 3, 0),
    (7, 2, 2, 4): (110, 20, 0, 0),
    (7, 2, 4, 4): (110, 20, 3, 0),
    (7, 4, 2, 4): (120, 45, 0, 0),
    (7, 4, 4, 4): (120, 50, 3, 0),
    (8, 1, 4, 4): (120, 10, 1, 0),
    (8, 2, 2, 4): (120, 25, 0, 0),
    (8, 2, 4, 4): (120, 25, 3, 0),
    (8, 4, 2, 4): (140, 45, 0, 0),
    (8, 4, 4, 4): (130, 45, 3, 0),
    (12, 4, 2, 4): (150, 45, 0, 0),
    (12, 4, 4, 4): (150, 45, 3, 0),
}


@dataclass
class Target:
    case: Tuple[int, int, int, int]
    aut: Automaton
    flank: int                        # flank_length with a closed end band (band_closed == 1)
    flank_open: Optional[int]         # flank_length that opens the end band (band_closed == 0)
    locus: Optional[synth.SynthLocus] = None    # regex targets
    reverse: bool = False

    @property
    def mv(self) -> int:
        return self.case[3]

    @property
    def is_regex(self) -> bool:
        return self.locus is not None

    def automaton(self, quantised: bool = False) -> Automaton:
        return self.aut.quantised() if quantised else self.aut

    def reads(self, n: int, seed: int, quantised: bool = False, noise: float = NOISE) -> List[np.ndarray]:
        """``n`` reads: every state held for at least mv samples, one stall of 40-200 samples of a
        single state, Gaussian noise; quantised: levels and samples on the 1/8 grid."""
        rng = np.random.default_rng([seed, 0x1A7, int(quantised)] + list(self.case))
        aut = self.automaton(quantised)
        out = []
        for _ in range(n):
            levels = self._regex_levels(rng) if self.is_regex else self._walk_levels(rng, aut)
            if quantised:
                levels = np.round(levels / QUANTUM) * QUANTUM
            p = int(rng.integers(len(levels) // 4, 3 * len(levels) // 4))
            levels = np.concatenate([levels[:p], np.full(int(rng.integers(40, 201)), levels[p]), levels[p:]])
            x = levels + rng.normal(0.0, noise, len(levels))
            out.append(np.round(x / QUANTUM) * QUANTUM if quantised else x)
        return out

    def _regex_levels(self, rng) -> np.ndarray:
        seq = self.locus.left + synth.draw_allele(rng, self.locus.units) + self.locus.right
        if self.reverse:
            seq = reverse_complement(seq)
        return synth.squiggle(rng, seq, get_pore_model(), noise=0.0, dwell=(self.mv, self.mv + 9))

    def _walk_levels(self, rng, aut: Automaton) -> np.ndarray:
        """A random path from state 0 to the end state (at most two rounds of the back edge), each state
        held mv or more samples, about 3 000 samples in all."""
        S, ip, ii = aut.n_states, aut.in_ptr, aut.in_idx
        succ = [[] for _ in range(S)]
        for j in range(S):
            for q in ii[ip[j]:ip[j + 1]]:
                succ[int(q)].append(j)
        live = np.zeros(S, dtype=bool)         # states the end state can be reached from
        live[aut.endstate] = True
        stack = [aut.endstate]
        while stack:
            j = stack.pop()
            for q in ii[ip[j]:ip[j + 1]]:
                if not live[q]:
                    live[q] = True
                    stack.append(int(q))
        path, j, loops = [0], 0, 0
        while j != aut.endstate:
            nxt = [t for t in succ[j] if live[t] and (t > j or loops < 2)]
            t = int(rng.choice(nxt))
            loops += t < j
            path.append(t)
            j = t
        mean = max(self.mv + 4.5, 3000.0 / len(path))
        dwell = self.mv + rng.integers(0, int(2 * (mean - self.mv)) + 1, len(path))
        return np.repeat(aut.values[path], dwell)


def _open_flank(aut: Automaton, flank: int) -> Optional[int]:
    for f in range(flank + 1, flank + 40):
        if not aut.band_closed(f):
            return f
    return None


def target(case) -> Target:
    if case in REGEX:
        name, flank, reverse = REGEX[case]
        locus = synth.make_locus(name, seed=3, flank_length=flank)
        aut = _regex_automaton(StateAutomata(locus.reverse_regex if reverse else locus.template_regex))
        return Target(case, aut, flank, _open_flank(aut, flank), locus, reverse)
    flank, positions, merges, comb = LADDER[case]
    aut = ladder(flank, positions, merges, comb)
    # flank_length = right chain: the band skips all but its last flank-10 states; one position past
    # the middle of the ladder opens it (the back edge leads from a kept state into a skipped one)
    return Target(case, aut, flank, flank + 10 + positions // 2)


_TARGETS = {}


def get(case) -> Target:
    if case not in _TARGETS:
        _TARGETS[case] = target(case)
    return _TARGETS[case]


def case_id(case) -> str:
    return 'kc{}_kg{}_deg{}_mv{}'.format(*case)


# ---------------------------------------------------------------------------------------------------
# layout invariants of a host plan (wstr_automaton_plan)
# ---------------------------------------------------------------------------------------------------
def assert_layout_invariants(in_ptr, in_idx, n_states: int, info: dict, sop: np.ndarray, what=None) -> None:
    """What wstr_automaton_create relies on: every state placed once, a generic slot's candidates cover
    its state's in-degree, chain slots hold chain links, and everything another lane reads is published."""
    in_ptr, in_idx = np.asarray(in_ptr), np.asarray(in_idx)
    KC, KG = info['chain_slots'], info['generic_slots']
    K = KC + KG
    assert sorted(int(s) for s in sop if s >= 0) == list(range(n_states)), what
    pos = {int(s): p for p, s in enumerate(sop) if s >= 0}
    deg = np.diff(in_ptr)
    code = info['unrolled_in_degree']   # 2 / 4; 100 + d: "low" layout; 200 + 10a + b: "graded" layout

    def incoming(s):
        return in_idx[in_ptr[s]:in_ptr[s + 1]]

    def slot_deg(g):                    # candidates generic slot g is built with (dtw.cu: slot_deg)
        if code >= 200:
            return (code - 200) // 10 if g == KG - 1 else ((code - 200) % 10 if g == KG - 2 else 1)
        if code >= 100:
            return code - 100 if g == KG - 1 else 1
        return code
    for s, p in pos.items():
        u = p % K
        if u >= KC:
            assert deg[s] <= slot_deg(u - KC), (what, s, u, code)
    outdeg = np.bincount(in_idx, minlength=n_states)
    for s, p in pos.items():
        lane, u = divmod(p, K)
        if u >= KC:
            continue
        # a chain slot holds a state with at most one incoming edge ...
        assert deg[s] <= 1, (what, s)
        if u > 0:
            # ... which comes from the slot before it, and that state feeds nothing else
            pred = int(incoming(s)[0])
            assert pos[pred] == p - 1 and outdeg[pred] == 1, (what, s)
        elif deg[s] == 1:
            # slot 0 reads a published value: a generic state or another lane's tail
            pp = pos[int(incoming(s)[0])]
            assert pp % K >= KC or pp % K == KC - 1, (what, s)
    # every predecessor of a generic state is published as well
    for s, p in pos.items():
        if p % K >= KC:
            for q in incoming(s):
                pp = pos[int(q)]
                assert pp % K >= KC or pp % K == KC - 1, (what, s)
