"""-m gpu: the phone error breakdown (nbasr_edit_align, trainer.edit_align_cuda, Trainer.error_report, sweep --errors)
against the numpy oracle (oracle/edit_np.py), exactly on counts, ref_at, hyp_at and confusion: greedy and beam-12 hypotheses,
rows with hyp_len 0, targets_len 0 and all-blank decodes, tie-heavy small alphabets, backpointers in shared memory and in
`work`, refused rows, accumulation over calls, the engine's log-probs in both precisions, and the sweep columns."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import nb_asr_b200 as nb  # noqa: E402
from gpu_utils import DEV  # noqa: E402
from nb_asr_b200 import _lib, data, sweep  # noqa: E402
from nb_asr_b200.trainer import edit_align_cuda  # noqa: E402
from oracle import decode_np as D  # noqa: E402
from oracle import edit_np as E  # noqa: E402

V = 49


def dev(a, dt):
    return torch.as_tensor(a).to(DEV, dt).contiguous()


def decoder():
    return nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[0], verbose=False)


def make_decode_case(seed, B, T, tgt_lo, tgt_hi):
    """Log-probs that half follow a blank-separated spelling of the reference (so hypotheses hold hits, substitutions,
    deletions and insertions), with row 1 all blank (hyp_len 0) and row 2 without reference tokens."""
    rng = np.random.default_rng(seed)
    tl = rng.integers(tgt_lo, tgt_hi, B).astype(np.int64)
    tl[2] = 0
    S = int(tgt_hi - 1)
    tg = np.zeros((B, S), np.int32)
    out_len = rng.integers(T // 2, T + 1, B).astype(np.int64)
    out_len[0] = T
    logits = 2.5 * rng.standard_normal((B, T, V)).astype(np.float32)
    for b in range(B):
        tg[b, :tl[b]] = rng.integers(1, V, tl[b])
        for t in range(0, int(out_len[b]), 2):
            if tl[b]:
                logits[b, t, tg[b, t * int(tl[b]) // int(out_len[b])]] += 3.0
        logits[b, 1::2, 0] += 3.0
    logits[1, :, 0] += 50.0
    lp = torch.log_softmax(torch.from_numpy(logits), -1)
    return lp, out_len, tg, tl


def run(hyp, hyp_len, tg, tl, lut, v=V, confusion=None):
    out = edit_align_cuda(hyp, hyp_len, dev(tg, torch.int32), dev(tl, torch.int64), lut, v, confusion)
    torch.cuda.synchronize()
    return out


def assert_equal_oracle(got, ref, rows=None):
    rows = slice(None) if rows is None else rows
    for name in ('counts', 'ref_at', 'hyp_at'):
        g = getattr(got, name)[rows].cpu().numpy()
        r = getattr(ref, name)[rows]
        assert np.array_equal(g, r), (name, np.argwhere(g != r)[:8].tolist())
    assert np.array_equal(got.confusion.cpu().numpy().view(np.uint64), ref.confusion)


@pytest.mark.parametrize('B,T,tgt_lo,tgt_hi,beam', [
    (8, 125, 20, 50, None),
    (8, 125, 20, 50, 12),
    (64, 125, 20, 50, None),         # cfg 2 eval: 64 x 500 input frames
    (64, 125, 20, 50, 12),
    (32, 750, 150, 301, None),       # 32 x 3 000 input frames, S_b <= 300
])
def test_decoded_hyps_match_oracle(B, T, tgt_lo, tgt_hi, beam):
    lp, out_len, tg, tl = make_decode_case(B * 1000 + T + (beam or 0), B, T, tgt_lo, tgt_hi)
    tr = decoder()
    tr.decode(lp, torch.from_numpy(out_len), (None, (torch.from_numpy(tg), torch.from_numpy(tl))), beam_width=beam)
    hyp, hl, dist = (x.clone() for x in tr.last_hyp)
    got = run(hyp, hl, tg, tl, tr._lut)
    ref = E.edit_align_batch(hyp.cpu().numpy(), hl.cpu().numpy(), tg, tl, D.FOLD_LUT, V)
    assert_equal_oracle(got, ref)
    c = got.counts.cpu()
    assert torch.equal(c[:, 1:].sum(1), dist.cpu())                 # S + D + I = greedy_per's / beam_per's dist
    assert int(hl[1]) == 0 and c[1, 0] == 0 and c[1, 1] == 0 and c[1, 3] == 0
    assert c[2].tolist() == [0, 0, 0, int(hl[2])]
    assert int(c[:, 0].sum()) > 0 and int(c[:, 1].sum()) > 0 and int(c[:, 2].sum()) > 0 and int(c[:, 3].sum()) > 0
    again = run(hyp, hl, tg, tl, tr._lut)
    for x, y in zip(got, again):
        assert torch.equal(x, y)


def random_rows(rng, B, H, S, alphabet, fold):
    hl = rng.integers(0, H + 1, B).astype(np.int32)
    tl = rng.integers(0, S + 1, B).astype(np.int64)
    h = rng.integers(1, alphabet + 1, (B, H))
    hyp = (D.FOLD_LUT[h] if fold else h).astype(np.int32)        # the fold maps no phone to 0
    tg = rng.integers(1, alphabet + 1, (B, S)).astype(np.int32)  # entries past the lengths are not read
    hl[0], tl[1] = 0, 0
    return hyp, hl, tg, tl


@pytest.mark.parametrize('alphabet,v', [(2, 3), (3, 4), (3, V)])
def test_small_alphabet_ties(alphabet, v):
    rng = np.random.default_rng(alphabet * 100 + v)
    hyp, hl, tg, tl = random_rows(rng, 64, 40, 40, alphabet, False)
    got = run(dev(hyp, torch.int32), dev(hl, torch.int32), tg, tl, None, v)
    assert_equal_oracle(got, E.edit_align_batch(hyp, hl, tg, tl, None, v))


@pytest.mark.parametrize('H,S,in_work', [(750, 300, False), (3000, 300, True), (1200, 1100, True)])
def test_backpointer_storage(H, S, in_work):
    lib = _lib.load()
    B = 4
    assert (lib.nbasr_edit_align_work_bytes(B, H, S) > 0) == in_work
    rng = np.random.default_rng(H + S)
    hyp, hl, tg, tl = random_rows(rng, B, H, S, 48, True)
    hl[2], tl[2] = H, S                                  # full length in both
    hl[3], tl[3] = H // 3, S                             # deletion-heavy
    lut = dev(D.FOLD_LUT, torch.int32)
    got = run(dev(hyp, torch.int32), dev(hl, torch.int32), tg, tl, lut)
    assert_equal_oracle(got, E.edit_align_batch(hyp, hl, tg, tl, D.FOLD_LUT, V))


def test_refused_rows_and_accumulation():
    rng = np.random.default_rng(9)
    hyp, hl, tg, tl = random_rows(rng, 10, 60, 40, 48, True)
    hl[:] = np.maximum(hl, 1)
    tl[:] = np.maximum(tl, 1)
    hyp[3, 0] = V                 # hyp id out of range
    hyp[4, hl[4] - 1] = 0         # a blank inside the hypothesis
    tg[6, 0] = V                  # target ids out of range
    tg[7, tl[7] - 1] = -2
    lut = dev(D.FOLD_LUT, torch.int32)
    conf = torch.zeros((V, V), dtype=torch.int64, device=DEV)
    got = run(dev(hyp, torch.int32), dev(hl, torch.int32), tg, tl, lut, confusion=conf)
    ref = E.edit_align_batch(hyp, hl, tg, tl, D.FOLD_LUT, V)
    for b in (3, 4, 6, 7):
        assert (got.counts[b] == -1).all() and (got.ref_at[b] == -1).all() and (got.hyp_at[b] == -1).all()
    assert_equal_oracle(got, ref)
    ok = [b for b in range(10) if b not in (3, 4, 6, 7)]
    clean = E.edit_align_batch(hyp[ok], hl[ok], tg[ok], tl[ok], D.FOLD_LUT, V)
    assert np.array_equal(ref.confusion, clean.confusion)
    # a second call adds into the same buffer
    again = run(dev(hyp, torch.int32), dev(hl, torch.int32), tg, tl, lut, confusion=conf)
    assert again.confusion is conf
    assert np.array_equal(conf.cpu().numpy().view(np.uint64), 2 * ref.confusion)
    assert torch.equal(again.counts, got.counts)
    with pytest.raises(ValueError):
        run(dev(hyp, torch.int32), dev(hl, torch.int32), tg, tl, lut, confusion=conf.float())


def test_shape_errors():
    one = torch.ones((1, 1), dtype=torch.int32, device=DEV)
    ln = torch.ones(1, dtype=torch.int32, device=DEV)
    tl = torch.ones(1, dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.NbasrError, match='64'):
        edit_align_cuda(one, ln, one, tl, None, 65)
    big = torch.ones((1, 32768), dtype=torch.int32, device=DEV)
    with pytest.raises(_lib.NbasrError, match='32768'):
        edit_align_cuda(big, ln, one, tl, None, V)
    with pytest.raises(_lib.NbasrError, match='shared memory'):
        edit_align_cuda(one, ln, torch.ones((1, 32767), dtype=torch.int32, device=DEV), tl, None, V)
    got = edit_align_cuda(one, ln, one, tl, None, V)        # hyp [1] against ref [1]
    assert got.counts.cpu().tolist() == [[1, 0, 0, 0]] and int(got.confusion[1, 1]) == 1


def trainer(arch, precision):
    nb.set_seed(1235)
    model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision=precision).eval()
    tr = decoder()
    tr.model = tr._model = model
    return tr


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_error_report_on_engine_logprobs(precision):
    tr = trainer([[4, 1], [4, 1, 1], [4, 1, 1, 1]], precision)          # c7d2_skips
    batch = nb.data.make_batch(16, 300, seed=3, min_len=100, tgt_lo=5, tgt_hi=40)
    _, logp, out_len = tr.step(batch, training=False)
    (_, _), (tg, tl) = batch
    for beam in (None, 12):
        per = tr.decode(logp, out_len, batch, beam_width=beam)
        hyp, hl, dist = (x.clone() for x in tr.last_hyp)
        rep = tr.error_report(logp, out_len, batch, beam_width=beam)
        assert torch.equal(rep.per, per)
        assert all(torch.equal(x, y) for x, y in zip(tr.last_hyp, (hyp, hl, dist)))
        assert torch.equal(rep.counts[:, 1:].sum(1).cpu(), dist.cpu())
        if beam is None:          # the numpy decode of the same log-probs gives the same folded hypotheses
            _, rd, _, fh = D.per_batch(logp.cpu().numpy(), out_len.cpu().numpy(), tg.numpy(), tl.numpy())
            assert dist.cpu().tolist() == rd.tolist()
            assert [hyp[b, :hl[b]].cpu().tolist() for b in range(16)] == [h.tolist() for h in fh]
        ref = E.edit_align_batch(hyp.cpu().numpy(), hl.cpu().numpy(), tg.numpy(), tl.numpy(), D.FOLD_LUT, V)
        assert_equal_oracle(rep, ref)
    bad = (batch[0], (tg.clone(), tl))
    bad[1][0][1, 0] = V
    with pytest.raises(ValueError):
        tr.error_report(logp, out_len, bad)


def test_sweep_error_columns():
    batches = data.timit_shaped_eval_set(n_utt=64, batch_size=32, seed=0)
    n_ref = sum(int(tl.sum()) for _, (t, tl) in batches)
    dev_batches = [((a.to(DEV), al.to(DEV)), (t.to(DEV), tl.to(DEV))) for (a, al), (t, tl) in batches]
    default = [[1, 0], [1, 0, 0], [1, 0, 0, 0]]
    kw = dict(seed=1235, init='device', conv_gain=101 ** 0.5, n_ref=n_ref)
    plain = sweep.evaluate_arch(default, dev_batches, 0, 'bf16', **kw)
    row = sweep.evaluate_arch(default, dev_batches, 0, 'bf16', errors=True, **kw)
    assert set(plain) == {'arch', 'loss', 'per', 'per_corpus'}
    assert set(row) == set(plain) | set(sweep.ERROR_COLUMNS)
    assert row['per'] == pytest.approx(plain['per'], abs=1e-12)
    assert row['per_corpus'] == pytest.approx(plain['per_corpus'], abs=1e-12)
    # sum over the corpus of S + D + I equals the sum of the decode's edit distances
    errs = sum(row[c] for c in sweep.ERROR_COLUMNS) * n_ref
    assert round(errs) == round(row['per_corpus'] * n_ref) and abs(errs - round(errs)) < 1e-6
    assert all(row[c] >= 0 for c in sweep.ERROR_COLUMNS) and errs > 0
