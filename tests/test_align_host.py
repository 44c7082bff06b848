"""CPU: the CTC forced-alignment oracle (oracle/align_np.py) against brute force and torchaudio, its edge cases, and the
ABI table entry of nbasr_ctc_align."""
import itertools
import warnings

import numpy as np
import pytest

from nb_asr_b200 import _lib
from oracle import align_np as A


def brute_force(lp, y):
    """Every frame-label sequence over V classes that collapses to y: (max sequential fp32 score, labels of the maximum
    picked by the tie rule) or (-inf, None).  The tie rule in path terms: among the best paths, the one whose state
    sequence read from the last frame backwards is lexicographically largest (trailing blank before the last label,
    then stay before s-1 before s-2)."""
    T, V = lp.shape
    S = len(y)
    seqs = np.array(list(itertools.product(range(V), repeat=T)), dtype=np.int64)
    prev = np.concatenate([np.full((len(seqs), 1), -1), seqs[:, :-1]], axis=1)
    kept = (seqs != 0) & (seqs != prev)
    n = np.cumsum(kept, axis=1)
    ok = n[:, -1] == S
    if S:
        ypad = np.asarray(y, np.int64)[np.clip(n - 1, 0, S - 1)]
        ok &= np.all(~kept | (seqs == ypad), axis=1)
    if not ok.any():
        return np.float32(-np.inf), None
    seqs, n = seqs[ok], n[ok]
    acc = np.zeros(len(seqs), np.float32)
    for t in range(T):
        acc = (acc + lp[t, seqs[:, t]]).astype(np.float32)
    best = acc.max()
    win = acc == best
    states = (2 * n - (seqs != 0))[win]
    order = np.lexsort([states[:, t] for t in range(T)])
    return best, seqs[win][order[-1]]


def random_targets(rng, S, V, p_repeat=0.4):
    y = []
    for _ in range(S):
        y.append(y[-1] if y and rng.random() < p_repeat else int(rng.integers(1, V)))
    return y


def one(lp, y, Tb=None):
    T, V = lp.shape
    tg = np.zeros((1, max(1, len(y))), np.int32)
    tg[0, :len(y)] = y
    return A.ctc_align(lp[None], [T if Tb is None else Tb], tg, [len(y)])


@pytest.mark.parametrize('quantised', [True, False])
def test_oracle_matches_brute_force(quantised):
    rng = np.random.default_rng(7 if quantised else 8)
    V = 5
    ties = 0
    for case in range(60):
        T = int(rng.integers(1, 8))
        S = int(rng.integers(0, 4))
        y = random_targets(rng, S, V)
        if quantised:      # multiples of 0.5: every sum is exact and equal path scores are common
            lp = (-0.5 * rng.integers(0, 5, size=(T, V))).astype(np.float32)
        else:
            lp = rng.standard_normal((T, V)).astype(np.float32) - 2.0
        best, path = brute_force(lp, y)
        got = one(lp, y)
        assert got.score[0] == best, (case, T, y)
        if path is None:
            assert (got.labels == -1).all()
            continue
        ties += int(got.tied[0])
        if quantised:
            np.testing.assert_array_equal(got.labels[0], path, err_msg=f'case {case}: T={T} y={y}')
        acc = np.float32(0)
        for t in range(T):
            acc = np.float32(acc + lp[t, got.labels[0, t]])
        assert acc == got.score[0]
    if quantised:
        assert ties > 10          # the tie rule was exercised


def test_oracle_matches_torchaudio():
    ta = pytest.importorskip('torchaudio')
    import torch
    rng = np.random.default_rng(11)
    V = 49
    done = 0
    while done < 40:
        T = int(rng.integers(20, 201))
        S = int(rng.integers(1, T // 3))
        y = random_targets(rng, S, V, p_repeat=0.2)
        logits = 3.0 * rng.standard_normal((T, V)).astype(np.float32)
        lp = torch.log_softmax(torch.from_numpy(logits), -1).numpy()
        got = one(lp, y)
        if got.tied[0]:
            continue
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ali, sc = ta.functional.forced_align(torch.from_numpy(lp)[None], torch.tensor([y], dtype=torch.int32), blank=0)
        np.testing.assert_array_equal(got.labels[0], ali[0].numpy())
        ref = float(sc[0].double().sum())
        assert abs(float(got.score[0]) - ref) <= 1e-5 * abs(ref)
        done += 1


def test_invariants_and_spans():
    rng = np.random.default_rng(3)
    B, T, S, V = 16, 60, 20, 49
    tl = rng.integers(0, S + 1, B)
    alen = rng.integers(0, 4 * T + 1, B)
    tg = np.zeros((B, S), np.int32)
    for b in range(B):
        tg[b, :tl[b]] = random_targets(rng, int(tl[b]), V)
    lp = torch_free_log_softmax(rng.standard_normal((B, T, V)).astype(np.float32))
    r = A.ctc_align(lp, alen, tg, tl, len_div=4)
    for b in range(B):
        Tb, Sb = min(T, alen[b] // 4), int(tl[b])
        assert (r.labels[b, Tb:] == -1).all() and (r.tok[b, Tb:] == -1).all()
        assert (r.start[b, Sb:] == -1).all() and (r.end[b, Sb:] == -1).all()
        if r.score[b] == -np.inf:
            assert (r.labels[b] == -1).all() and (r.start[b] == -1).all()
            continue
        assert A.collapse(r.labels[b, :Tb]) == tg[b, :Sb].tolist()
        for j in range(Sb):
            span = np.nonzero(r.tok[b] == j)[0]
            assert r.start[b, j] == span[0] and r.end[b, j] == span[-1] + 1 == r.start[b, j] + len(span)
            assert (r.labels[b, span] == tg[b, j]).all()
        assert ((r.tok[b, :Tb] == -1) == (r.labels[b, :Tb] == 0)).all()


def torch_free_log_softmax(x):
    m = x.max(-1, keepdims=True)
    return (x - m - np.log(np.exp(x - m).sum(-1, keepdims=True))).astype(np.float32)


def test_edge_cases():
    rng = np.random.default_rng(5)
    lp = torch_free_log_softmax(rng.standard_normal((6, 5)).astype(np.float32))
    # infeasible: two frames cannot hold a repeated label (it needs a blank in between); three can
    assert one(lp[:2], [2, 2]).score[0] == -np.inf
    assert (one(lp[:2], [2, 2]).labels == -1).all() and (one(lp[:2], [2, 2]).end == -1).all()
    r = one(lp[:3], [2, 2])
    assert r.labels[0].tolist() == [2, 0, 2] and r.start[0].tolist() == [0, 2] and r.end[0].tolist() == [1, 3]
    # no frames: infeasible with tokens, score 0 without
    assert one(lp, [1], Tb=0).score[0] == -np.inf
    r = one(lp, [], Tb=0)
    assert r.score[0] == 0 and (r.labels == -1).all()
    # S_b = 0: the all-blank path
    r = one(lp, [])
    assert (r.labels[0] == 0).all() and (r.tok[0] == -1).all()
    acc = np.float32(0)
    for t in range(6):
        acc = np.float32(acc + lp[t, 0])
    assert r.score[0] == acc
    # T_b = 1 with one token: the label itself
    r = one(lp, [3], Tb=1)
    assert r.labels[0].tolist() == [3, -1, -1, -1, -1, -1] and r.score[0] == lp[0, 3]
    assert r.start[0].tolist() == [0] and r.end[0].tolist() == [1]
    # T_b < T: frames past the length are -1
    r = one(lp, [1, 4], Tb=4)
    assert (r.labels[0, 4:] == -1).all() and (r.labels[0, :4] >= 0).all()
    with pytest.raises(ValueError):
        one(lp, [1, 5])


def test_align_in_abi_table():
    assert 'nbasr_ctc_align' in _lib.EXPORTS and 'nbasr_ctc_align_work_bytes' in _lib.EXPORTS
