"""CPU: the phone-error-breakdown oracle (oracle/edit_np.py) against brute-force enumeration of every alignment, its
invariants and edge cases, the SURVEY KAT, the batch form (fold, refused rows, confusion), and the sweep's --errors flag."""
import itertools

import numpy as np
import pytest

from nb_asr_b200 import _lib, sweep
from oracle import decode_np as Dn
from oracle import edit_np as E


def all_alignments(n, m):
    """Every move sequence from (n, m) back to (0, 0), read from the end: DIAG (i-1, j-1), DEL (j-1), INS (i-1)."""
    if n == 0 and m == 0:
        yield ()
        return
    if n and m:
        for rest in all_alignments(n - 1, m - 1):
            yield (E.DIAG,) + rest
    if m:
        for rest in all_alignments(n, m - 1):
            yield (E.DEL,) + rest
    if n:
        for rest in all_alignments(n - 1, m):
            yield (E.INS,) + rest


def cost(hyp, ref, moves):
    i, j, c = len(hyp), len(ref), 0
    for mv in moves:
        if mv == E.DIAG:
            i, j = i - 1, j - 1
            c += hyp[i] != ref[j]
        elif mv == E.DEL:
            j, c = j - 1, c + 1
        else:
            i, c = i - 1, c + 1
    return c


def check_invariants(hyp, ref, a):
    hits, subs, dels, ins = (int(x) for x in a.counts)
    assert hits + subs + dels == len(ref) and hits + subs + ins == len(hyp)
    assert subs + dels + ins == Dn.levenshtein(hyp, ref)
    paired = [(i, int(j)) for i, j in enumerate(a.ref_at) if j >= 0]
    assert paired == [(int(i), j) for j, i in enumerate(a.hyp_at) if i >= 0]      # the two maps are inverse
    assert all(j1 < j2 for (_, j1), (_, j2) in zip(paired, paired[1:]))           # monotone
    assert sum(hyp[i] == ref[j] for i, j in paired) == hits
    assert int((a.ref_at < 0).sum()) == ins and int((a.hyp_at < 0).sum()) == dels


@pytest.mark.parametrize('alphabet', [2, 3])
def test_oracle_matches_brute_force(alphabet):
    rng = np.random.default_rng(alphabet)
    ties = 0
    for case in range(150):
        n, m = (int(x) for x in rng.integers(0, 6, 2))
        hyp = [int(x) for x in rng.integers(1, alphabet + 1, n)]
        ref = [int(x) for x in rng.integers(1, alphabet + 1, m)]
        costs = {mv: cost(hyp, ref, mv) for mv in all_alignments(n, m)}
        best = min(costs.values())
        optimal = sorted(mv for mv, c in costs.items() if c == best)
        ties += len(optimal) > 1
        a = E.edit_align(hyp, ref)
        assert best == Dn.levenshtein(hyp, ref) == cost(hyp, ref, a.moves), (case, hyp, ref)
        assert tuple(a.moves) == optimal[0], (case, hyp, ref, a.moves, optimal[:3])
        check_invariants(hyp, ref, a)
    assert ties > 50              # the tie rule was exercised


def test_exhaustive_small():
    """Every pair over {1, 2} with |hyp|, |ref| <= 4."""
    for n, m in itertools.product(range(5), repeat=2):
        for hyp in itertools.product((1, 2), repeat=n):
            for ref in itertools.product((1, 2), repeat=m):
                a = E.edit_align(hyp, ref)
                costs = {mv: cost(hyp, ref, mv) for mv in all_alignments(n, m)}
                best = min(costs.values())
                assert tuple(a.moves) == min(mv for mv, c in costs.items() if c == best)


def test_empty_sequences():
    a = E.edit_align([], [])
    assert a.counts.tolist() == [0, 0, 0, 0] and a.moves == []
    a = E.edit_align([], [4, 5, 4])
    assert a.counts.tolist() == [0, 0, 3, 0] and a.hyp_at.tolist() == [-1, -1, -1] and len(a.ref_at) == 0
    a = E.edit_align([4, 5], [])
    assert a.counts.tolist() == [0, 0, 0, 2] and a.ref_at.tolist() == [-1, -1] and len(a.hyp_at) == 0


def test_survey_kat():
    hyp, ref = [11, 9, 20, 20, 5, 14], [19, 9, 20, 20, 9, 14, 7]
    a = E.edit_align(hyp, ref)
    assert a.counts.tolist() == [4, 2, 1, 0]            # hits, substitutions, deletions (the trailing 7), insertions
    assert a.hyp_at.tolist() == [0, 1, 2, 3, 4, 5, -1]
    assert a.ref_at.tolist() == [0, 1, 2, 3, 4, 5]
    check_invariants(hyp, ref, a)


def test_tie_rule_examples():
    # hyp [1] against ref [2, 1]: the hit on the last ref token beats deleting it
    assert E.edit_align([1], [2, 1]).hyp_at.tolist() == [-1, 0]
    # hyp [1, 2] against ref [3]: 2 -> 3 with 1 inserted, or 1 -> 3 with 2 inserted (cost 2 each); the diagonal from
    # (2, 1) comes first
    assert E.edit_align([1, 2], [3]).ref_at.tolist() == [-1, 0]
    # hyp [1] against ref [2]: substitution (cost 1) beats deletion + insertion (cost 2)
    assert E.edit_align([1], [2]).counts.tolist() == [0, 1, 0, 0]
    # hyp [3] against ref [1, 2]: diagonal (3 -> 2) then deletion of 1, not deletion of 2
    assert E.edit_align([3], [1, 2]).hyp_at.tolist() == [-1, 0]


def test_batch_form():
    rng = np.random.default_rng(4)
    B, H, S, V = 12, 30, 20, 49
    hyp = np.zeros((B, H), np.int32)
    hl = rng.integers(0, H + 1, B).astype(np.int32)
    tg = rng.integers(1, V, (B, S)).astype(np.int32)
    tl = rng.integers(0, S + 1, B).astype(np.int64)
    for b in range(B):
        hyp[b, :hl[b]] = Dn.FOLD_LUT[rng.integers(1, V, hl[b])]
        hyp[b, :hl[b]][hyp[b, :hl[b]] == 0] = 1
    tg[3, 2] = 0                      # a zero token inside the reference is dropped, like greedy_per does
    hl[5], tl[6] = 0, 0
    hyp[7, 0] = V                     # refused rows: hyp id out of range, target id out of range
    hl[7] = max(hl[7], 1)
    tg[8, 0], tl[8] = -1, max(tl[8], 1)
    r = E.edit_align_batch(hyp, hl, tg, tl, Dn.FOLD_LUT, V)
    for b in range(B):
        if b in (7, 8):
            assert (r.counts[b] == -1).all() and (r.ref_at[b] == -1).all() and (r.hyp_at[b] == -1).all()
            continue
        ref = E.compared_ref(tg[b], tl[b], Dn.FOLD_LUT)
        a = E.edit_align(hyp[b, :hl[b]], ref)
        assert (r.counts[b] == a.counts).all()
        assert (r.ref_at[b, hl[b]:] == -1).all() and (r.hyp_at[b, len(ref):] == -1).all()
        check_invariants(hyp[b, :hl[b]].tolist(), ref.tolist(), a)
    ok = [b for b in range(B) if b not in (7, 8)]
    c = r.counts[ok].sum(0)
    assert int(r.confusion.sum()) == int(c.sum())
    assert int(r.confusion[0].sum()) == c[3] and int(r.confusion[:, 0].sum()) == c[2]
    assert int(np.trace(r.confusion)) == c[0]
    assert len(E.compared_ref(tg[3], S, Dn.FOLD_LUT)) == S - 1


def test_sweep_errors_flag():
    assert sweep.build_parser().parse_args(['--errors']).errors is True
    assert sweep.build_parser().parse_args([]).errors is False
    assert sweep.ERROR_COLUMNS == ('sub_rate', 'del_rate', 'ins_rate')


def test_edit_align_in_abi_table():
    assert 'nbasr_edit_align' in _lib.EXPORTS and 'nbasr_edit_align_work_bytes' in _lib.EXPORTS
    lib = _lib.load()
    assert lib.nbasr_edit_align_work_bytes(64, 125, 49) == 0 and lib.nbasr_edit_align_work_bytes(32, 750, 300) == 0
    assert lib.nbasr_edit_align_work_bytes(4, 3000, 300) == 4 * 8 * 3301 * 10
