"""-m gpu: CTC forced alignment (nbasr_ctc_align, trainer.ctc_align_cuda, Trainer.align) against the numpy fp32 oracle
(oracle/align_np.py), bit-exact on all five outputs: mixed lengths, repeats, rows without a path, S_b = 0 and T_b = 0 in
one batch; quantised log-probs for ties; backpointers in shared memory and in `work`; errors; the engine's log-probs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import nb_asr_b200 as nb  # noqa: E402
from gpu_utils import DEV  # noqa: E402
from nb_asr_b200 import _lib  # noqa: E402
from nb_asr_b200.trainer import ctc_align_cuda  # noqa: E402
from oracle import align_np as A  # noqa: E402

V = 49


def make_case(seed, B, T, S, len_div, quantised):
    """Rows cycle through: random lengths, many repeats, no path (S_b > T_b), S_b = 0, T_b = 0 with tokens; row 0 has
    T_b = T."""
    rng = np.random.default_rng(seed)
    if quantised:           # multiples of 0.5: exact sums, many equal candidates
        lp = (-0.5 * rng.integers(0, 6, size=(B, T, V))).astype(np.float32)
    else:
        x = 3.0 * rng.standard_normal((B, T, V)).astype(np.float32)
        lp = torch.log_softmax(torch.from_numpy(x), -1).numpy()
    Tb = rng.integers(1, T + 1, B)
    Tb[0] = T
    tl = np.zeros(B, np.int64)
    tg = np.zeros((B, S), np.int32)
    for b in range(B):
        kind = b % 5
        n = int(rng.integers(1, min(S, max(1, int(Tb[b]) // 2)) + 1))      # n + repeats <= 2n - 1 < T_b: a path exists
        if kind == 2:                                                       # more tokens than frames
            n = S
            Tb[b] = min(int(Tb[b]), S // 2)
        elif kind == 3:
            n = 0
        elif kind == 4:
            Tb[b] = 0
        y = []
        for _ in range(n):
            y.append(y[-1] if y and rng.random() < (0.9 if kind == 1 else 0.2) else int(rng.integers(1, V)))
        tg[b, :n] = y
        tl[b] = n
    alen = Tb * len_div + rng.integers(0, len_div, B)      # the kernel divides: remainders must not matter
    return lp, alen.astype(np.int64), tg, tl


def run(lp, alen, tg, tl, len_div):
    t = lambda a, dt: torch.as_tensor(a).to(DEV, dt).contiguous()   # noqa: E731
    out = ctc_align_cuda(t(lp, torch.float32), t(alen, torch.int64), len_div, t(tg, torch.int32), t(tl, torch.int64))
    torch.cuda.synchronize()
    return out


def assert_equal_oracle(got, ref, rows=None):
    rows = slice(None) if rows is None else rows
    for name in ('labels', 'tok', 'start', 'end', 'score'):
        g = getattr(got, name)[rows].cpu()
        r = torch.from_numpy(np.ascontiguousarray(getattr(ref, name)[rows]))
        assert torch.equal(g, r), (name, torch.nonzero(g != r)[:8].tolist())


def check_invariants(got, lp, tg, tl, alen, len_div):
    labels, tok, start, end, score = (x.cpu().numpy() for x in got)
    B, T = labels.shape
    feasible = 0
    for b in range(B):
        Tb, Sb = min(T, int(alen[b]) // len_div), int(tl[b])
        if score[b] == -np.inf:
            continue
        feasible += 1
        assert A.collapse(labels[b, :Tb]) == tg[b, :Sb].tolist()
        for j in range(Sb):
            span = np.nonzero(tok[b] == j)[0]
            assert start[b, j] == span[0] and end[b, j] == span[-1] + 1 == start[b, j] + len(span)
        acc = np.float32(0)
        for t in range(Tb):
            acc = np.float32(acc + lp[b, t, labels[b, t]])
        assert acc.tobytes() == score[b].tobytes()
    return feasible


@pytest.mark.parametrize('B,T,S,len_div,quantised', [
    (1, 40, 12, 1, False),
    (7, 200, 60, 4, True),
    (64, 125, 49, 1, False),        # cfg 2 eval: 64 x 500 input frames
    (64, 125, 49, 4, True),
    (7, 750, 300, 1, False),        # cfg 5 worst case, L = 601: backpointers in shared memory
    (7, 1500, 300, 4, True),        # backpointers in `work`
])
def test_kernel_matches_oracle(B, T, S, len_div, quantised):
    lib = _lib.load()
    assert (lib.nbasr_ctc_align_work_bytes(B, T, S) > 0) == (T >= 1500)
    lp, alen, tg, tl = make_case(B * 1000 + T + S, B, T, S, len_div, quantised)
    ref = A.ctc_align(lp, alen, tg, tl, len_div)
    got = run(lp, alen, tg, tl, len_div)
    assert_equal_oracle(got, ref)
    if quantised:
        assert ref.tied.any()
    if B > 1:
        assert (ref.score == -np.inf).any() and (tl == 0).any()
    assert check_invariants(got, lp, tg, tl, alen, len_div) >= (B + 1) // 2
    again = run(lp, alen, tg, tl, len_div)
    for x, y in zip(got, again):
        assert torch.equal(x, y)


def test_errors():
    lp, alen, tg, tl = make_case(5, 6, 60, 10, 1, False)
    tg[tl == 0, 0] = 7
    tl[:] = np.maximum(tl, 1)
    tg[2, 0] = V                      # out of range: that row is refused on the device, the others are untouched
    tg[4, 0] = -3
    got = run(lp, alen, tg, tl, 1)
    score = got.score.cpu().numpy()
    assert np.isnan(score[[2, 4]]).all()
    for name in ('labels', 'tok', 'start', 'end'):
        assert (getattr(got, name)[[2, 4]] == -1).all()
    ok = [0, 1, 3, 5]
    tg_ok = tg.copy()
    tg_ok[[2, 4], 0] = 1
    assert_equal_oracle(got, A.ctc_align(lp, alen, tg_ok, tl), rows=ok)
    big = np.zeros((1, 512), np.int32) + 1
    with pytest.raises(_lib.NbasrError, match='exceeds'):
        run(lp[:1], alen[:1], big, np.array([512]), 1)
    run(lp[:1, :], np.array([60]), big[:, :511], np.array([20]), 1)      # S = 511 is the largest accepted


def trainer(arch, precision):
    nb.set_seed(1235)
    model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision=precision).eval()
    tr = nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[0], verbose=False)
    tr.model = tr._model = model
    return tr


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_trainer_align_on_engine_logprobs(precision):
    tr = trainer([[4, 1], [4, 1, 1], [4, 1, 1, 1]], precision)          # c7d2_skips
    batch = nb.data.make_batch(16, 300, seed=3, min_len=100, tgt_lo=5, tgt_hi=40)
    _, logp, out_len = tr.step(batch, training=False)
    ali = tr.align(logp, out_len, batch)
    torch.cuda.synchronize()
    (_, _), (tg, tl) = batch
    ref = A.ctc_align(logp.cpu().numpy(), out_len.cpu().numpy(), tg.numpy(), tl.numpy())
    assert_equal_oracle(ali, ref)
    assert np.isfinite(ref.score).sum() >= 8
    bad = (batch[0], (tg.clone(), tl))
    bad[1][0][1, 0] = V
    with pytest.raises(ValueError):
        tr.align(logp, out_len, bad)
