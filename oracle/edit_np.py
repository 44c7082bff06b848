"""numpy restatement of the phone error breakdown (nbasr_edit_align, include/nbasr.h).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Levenshtein table over the hypothesis (i) and the reference (j):
    D(i, 0) = i, D(0, j) = j, D(i, j) = min(D(i-1, j-1) + [hyp[i-1] != ref[j-1]], D(i, j-1) + 1, D(i-1, j) + 1)
so D(n, m) is decode_np.levenshtein(hyp, ref), the `dist` of nbasr_greedy_per.  ASR terms: a diagonal step is a hit or a
substitution, a step j-1 a deletion (ref token aligned to nothing), a step i-1 an insertion (hyp token aligned to nothing).
Tie rule: backtrace from (n, m) taking at each cell the first move that lies on an optimal path in the order diagonal,
deletion, insertion (on the borders the only move there is); equivalently, among all minimum-cost alignments the one
whose move sequence read from the end is lexicographically smallest under diagonal < deletion < insertion.
"""
import collections

import numpy as np

from .decode_np import FOLD_LUT, levenshtein  # noqa: F401  (FOLD_LUT: the `lut` of Trainer.error_report)

DIAG, DEL, INS = 0, 1, 2

Alignment = collections.namedtuple('Alignment', 'counts ref_at hyp_at moves')
Batch = collections.namedtuple('Batch', 'counts ref_at hyp_at confusion')


def edit_align(hyp, ref):
    """One pair of compared sequences -> Alignment: counts [hits, substitutions, deletions, insertions], ref_at (n,)
    ref position of each hyp position (-1: insertion), hyp_at (m,) hyp position of each ref position (-1: deletion),
    moves: the move sequence read from the end (DIAG / DEL / INS)."""
    hyp = [int(x) for x in hyp]
    ref = [int(x) for x in ref]
    n, m = len(hyp), len(ref)
    D = np.zeros((n + 1, m + 1), np.int64)
    D[:, 0] = np.arange(n + 1)
    D[0, :] = np.arange(m + 1)
    for i in range(1, n + 1):
        for j in range(1, m + 1):
            D[i, j] = min(D[i - 1, j - 1] + (hyp[i - 1] != ref[j - 1]), D[i, j - 1] + 1, D[i - 1, j] + 1)
    counts = [0, 0, 0, 0]
    ref_at = np.full(n, -1, np.int32)
    hyp_at = np.full(m, -1, np.int32)
    moves = []
    i, j = n, m
    while i > 0 or j > 0:
        if i > 0 and j > 0 and D[i - 1, j - 1] + (hyp[i - 1] != ref[j - 1]) == D[i, j]:
            i, j = i - 1, j - 1
            ref_at[i], hyp_at[j] = j, i
            counts[0 if hyp[i] == ref[j] else 1] += 1
            moves.append(DIAG)
        elif j > 0 and D[i, j - 1] + 1 == D[i, j]:
            j -= 1
            counts[2] += 1
            moves.append(DEL)
        else:
            i -= 1
            counts[3] += 1
            moves.append(INS)
    return Alignment(np.array(counts, np.int32), ref_at, hyp_at, moves)


def compared_ref(targets_row, targets_len, lut):
    """targets[:min(S, targets_len)] through lut (or as is), tokens that map to 0 dropped."""
    r = np.asarray(targets_row[:max(0, min(len(targets_row), int(targets_len)))], np.int64)
    if lut is not None:
        r = np.asarray(lut, np.int64)[r]
    return r[r != 0]


def edit_align_batch(hyp, hyp_len, targets, targets_len, lut, V):
    """What nbasr_edit_align computes for one call with a zero confusion matrix: hyp (B, H) / hyp_len (B,) as
    nbasr_greedy_per writes them, targets (B, S) / targets_len (B,), lut (V,) or None -> Batch(counts (B, 4) int32,
    ref_at (B, H) int32, hyp_at (B, S) int32, confusion (V, V) uint64).  Rows with a target id outside [0, V) (before or
    after lut) or a hyp id outside [1, V) are refused: -1 outputs, nothing added to confusion."""
    hyp, targets = np.asarray(hyp), np.asarray(targets)
    B, H = hyp.shape
    S = targets.shape[1]
    counts = np.full((B, 4), -1, np.int32)
    ref_at = np.full((B, H), -1, np.int32)
    hyp_at = np.full((B, S), -1, np.int32)
    conf = np.zeros((V, V), np.uint64)
    for b in range(B):
        h = hyp[b, :max(0, min(H, int(hyp_len[b])))].astype(np.int64)
        raw = targets[b, :max(0, min(S, int(targets_len[b])))].astype(np.int64)
        if np.any((h < 1) | (h >= V)) or np.any((raw < 0) | (raw >= V)):
            continue
        if lut is not None and np.any((np.asarray(lut)[raw] < 0) | (np.asarray(lut)[raw] >= V)):
            continue
        r = compared_ref(raw, len(raw), lut)
        a = edit_align(h, r)
        counts[b] = a.counts
        ref_at[b, :len(h)] = a.ref_at
        hyp_at[b, :len(r)] = a.hyp_at
        for i, j in enumerate(a.ref_at):
            conf[r[j] if j >= 0 else 0, h[i]] += 1
        for j in np.nonzero(a.hyp_at < 0)[0]:
            conf[r[j], 0] += 1
    return Batch(counts, ref_at, hyp_at, conf)
