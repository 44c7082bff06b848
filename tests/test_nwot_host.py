"""CPU: host side of the NASWOT proxy (`nwot`) -- the score, the kernel-matrix definition against N_A - Hamming, the
valid-frame rule against the model's frame rule, the --proxies flag and the C ABI of nbasr_gate_gram."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from nb_asr_b200 import _lib, proxies, sweep
from oracle import nwot_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_nwot_score_is_slogdet():
    rng = np.random.default_rng(0)
    X = rng.integers(0, 2, (6, 300))
    K = (X @ X.T + (1 - X) @ (1 - X).T).astype(np.uint64)
    assert proxies.nwot_score(K) == pytest.approx(np.linalg.slogdet(K.astype(np.float64))[1], rel=1e-12)
    assert proxies.nwot_score(K) == R.nwot_score(K)
    K[3], K[:, 3] = K[1], K[:, 1]           # a duplicated utterance: singular
    K[3, 3] = K[1, 1]
    assert proxies.nwot_score(K) == -np.inf


def test_kernel_is_units_minus_hamming_for_equal_lengths():
    rng = np.random.default_rng(1)
    B, T = 5, 9
    codes = [(0, rng.random((B, 16, T)) < 0.5), (2, rng.random((B, 8, (T + 1) // 2)) < 0.3)]
    alen = np.full(B, T)
    K = R.kernel_from_codes(codes, alen)
    flat = np.concatenate([m.reshape(B, -1) for _, m in codes], axis=1).astype(np.int64)
    NA = flat.shape[1]
    ham = (flat[:, None, :] != flat[None, :, :]).sum(2)
    np.testing.assert_array_equal(K, NA - ham)
    assert np.all(np.diag(K) == NA)
    assert np.all(np.linalg.eigvalsh(K) > -1e-6)          # PSD


def test_kernel_with_unequal_lengths_counts_common_frames():
    rng = np.random.default_rng(2)
    B, T = 4, 11
    m = rng.random((B, 3, T)) < 0.5
    alen = np.array([11, 7, 1, 4])
    K = R.kernel_from_codes([(0, m)], alen)
    for i in range(B):
        for j in range(B):
            n = min(alen[i], alen[j])
            assert K[i, j] == (m[i, :, :n] == m[j, :, :n]).sum()
    assert np.all(np.linalg.eigvalsh(K) > -1e-6)


def test_length_rule_matches_model_frame_rule():
    assert proxies.LEN_SHIFT == (0, 0, 1, 2)
    for T in range(1, 1001):
        t_blk, tt = [], T
        for s in (1, 1, 2, 2):                          # model.py: T -> (T + 1) // 2 at every stride-2 block
            tt = tt if s == 1 else (tt + 1) // 2
            t_blk.append(tt)
        for k in range(4):
            assert proxies.gate_frames(T, t_blk[k], proxies.LEN_SHIFT[k]) == t_blk[k]
            assert int(R.frames([T], t_blk[k], k)[0]) == t_blk[k]
        # a shorter utterance in a batch padded to T: ceil(len / 2^s) is its own frame count, capped at T_k
        for ln in (1, T // 3 + 1, T):
            for k in range(4):
                own = ln if k < 2 else ((ln + 1) // 2 if k == 2 else ((ln + 1) // 2 + 1) // 2)
                assert proxies.gate_frames(ln, t_blk[k], proxies.LEN_SHIFT[k]) == min(own, t_blk[k])


def test_sweep_accepts_nwot():
    assert 'nwot' in proxies.MEASURES
    a = sweep.build_parser().parse_args(['--proxies', 'nwot'])
    assert a.proxies == ('nwot',)
    a = sweep.build_parser().parse_args(['--proxies', 'grad_norm,snip,nwot'])
    assert a.proxies == ('grad_norm', 'snip', 'nwot')
    assert 'nwot' in sweep.build_parser().format_help()


def test_lib_table_has_the_gate_gram():
    assert 'nbasr_gate_gram' in _lib.EXPORTS and 'nbasr_gate_gram_work_elems' in _lib.EXPORTS


def test_gate_layer_layout_matches_c(tmp_path):
    prog = tmp_path / 'gl.c'
    prog.write_text('''#include <stdio.h>
#include <stddef.h>
#include "nbasr.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(nbasr_gate_layer), offsetof(nbasr_gate_layer, mask_rows),
         offsetof(nbasr_gate_layer, w), offsetof(nbasr_gate_layer, C), offsetof(nbasr_gate_layer, Tp),
         offsetof(nbasr_gate_layer, T), offsetof(nbasr_gate_layer, s), offsetof(nbasr_gate_layer, reserved));
  return 0;
}''')
    exe = tmp_path / 'gl'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), str(prog), '-o', str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    G = _lib.GateLayer
    assert got == [ctypes.sizeof(G), G.mask_rows.offset, G.w.offset, G.C.offset, G.Tp.offset, G.T.offset, G.s.offset,
                   G.reserved.offset]
