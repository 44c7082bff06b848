"""numpy fp32 restatement of CTC forced alignment (nbasr_ctc_align, include/nbasr.h).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Viterbi through the CTC trellis of the extended label sequence
(blank, y_0, blank, ..., y_{S_b-1}, blank), blank = 0:
    alpha_0(0) = logp[0, 0], alpha_0(1) = logp[0, y_0], every other state -inf;
    alpha_t(s) = max(alpha_{t-1}(s), alpha_{t-1}(s-1), alpha_{t-1}(s-2) [ext[s] != 0 and ext[s] != ext[s-2]]) + logp[t, ext[s]]
with the max taken exactly and ONE fp32 add per step, so the scores and paths of the CUDA kernel are reproduced bit for bit.
Tie rule: on exact equality the smaller jump wins (stay, then s-1, then s-2); at the end the trailing blank 2S_b wins over
the last label 2S_b - 1 unless the label is strictly better.  A row whose best score is -inf has no path (with finite
log-probs: T_b < S_b + number of adjacent repeats, or T_b = 0 < S_b); T_b = S_b = 0 has score 0 and no frames.
Outputs (-1 for frames t >= T_b, tokens j >= S_b and every output of a row without a path):
    labels (B, T) class of each frame on the best path, tok (B, T) target index the frame emits (-1 on blanks),
    start / end (B, S) half-open frame span of each token, score (B,) fp32,
    tied (B,) whether an exact tie was broken on the returned path (so a comparison with another implementation, whose
    tie rule may differ, can pick tie-free inputs).
"""
import collections

import numpy as np

Alignment = collections.namedtuple('Alignment', 'labels tok start end score tied')


def ctc_align(logp, audio_len, targets, targets_len, len_div=1):
    """logp (B, T, V) log-probs (taken as fp32), audio_len (B,), targets (B, S) int, targets_len (B,) -> Alignment.
    T_b = min(T, audio_len // len_div), S_b = min(S, targets_len).  A target id outside [1, V) raises ValueError."""
    logp = np.asarray(logp, dtype=np.float32)
    targets = np.asarray(targets)
    B, T, V = logp.shape
    S = targets.shape[1]
    labels = np.full((B, T), -1, np.int32)
    tok = np.full((B, T), -1, np.int32)
    start = np.full((B, S), -1, np.int32)
    end = np.full((B, S), -1, np.int32)
    score = np.zeros(B, np.float32)
    tied = np.zeros(B, bool)
    neg = np.float32(-np.inf)
    for b in range(B):
        Tb = max(0, min(T, int(audio_len[b]) // len_div))
        Sb = max(0, min(S, int(targets_len[b])))
        y = targets[b, :Sb].astype(np.int64)
        if np.any((y < 1) | (y >= V)):
            raise ValueError(f'row {b}: target id outside [1, {V})')
        L = 2 * Sb + 1
        ext = np.zeros(L, np.int64)
        ext[1::2] = y
        skip = np.zeros(L, bool)
        skip[3::2] = y[1:] != y[:-1]
        if Tb == 0:
            score[b] = 0.0 if Sb == 0 else neg
            continue
        lp = logp[b]
        alpha = np.full(L, neg, np.float32)
        alpha[:min(L, 2)] = lp[0, ext[:2]]
        move = np.zeros((Tb, L), np.int8)
        tie = np.zeros((Tb, L), bool)
        for t in range(1, Tb):
            c1 = np.concatenate([[neg], alpha[:-1]])
            c2 = np.where(skip, np.concatenate([[neg, neg], alpha[:-2]])[:L], neg)
            mx = np.maximum(np.maximum(alpha, c1), c2)
            tie[t] = ((alpha == mx).astype(int) + (c1 == mx) + (c2 == mx) >= 2) & (mx > neg)
            a = alpha.copy()
            m = np.zeros(L, np.int8)
            up = c1 > a
            a[up] = c1[up]
            m[up] = 1
            up = c2 > a
            a[up] = c2[up]
            m[up] = 2
            move[t] = m
            alpha = (a + lp[t, ext]).astype(np.float32)
        s = L - 1
        if L >= 2 and alpha[L - 2] > alpha[L - 1]:
            s = L - 2
        score[b] = alpha[s]
        if alpha[s] == neg:
            continue
        tied[b] = L >= 2 and alpha[L - 2] == alpha[L - 1]
        path = np.empty(Tb, np.int64)
        for t in range(Tb - 1, -1, -1):
            path[t] = s
            if t >= 1:
                tied[b] |= tie[t, s]
                s -= int(move[t, s])
        labels[b, :Tb] = ext[path]
        odd = (path & 1) == 1
        tok[b, :Tb] = np.where(odd, path >> 1, -1)
        for t in range(Tb):
            if odd[t]:
                j = path[t] >> 1
                if start[b, j] < 0:
                    start[b, j] = t
                end[b, j] = t + 1
    return Alignment(labels, tok, start, end, score, tied)


def collapse(labels):
    """CTC collapse of one frame-label row (merge repeats, drop blanks and -1 padding)."""
    out, prev = [], -1
    for c in labels:
        c = int(c)
        if c != prev and c > 0:
            out.append(c)
        prev = c
    return out
