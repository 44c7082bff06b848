"""-m gpu: the NASWOT proxy (`nwot`, nb_asr_b200.proxies) -- nbasr_gate_gram against a torch bit-unpacking reference
(exact), K from a plan's own gate masks, K and the score against the fp64 CPU oracle (oracle/nwot_ref.py), and what
compute_proxies / the sweep must keep.  Oracle fixture: B x T = 8 x 200, as in test_gpu_10_proxies.py."""
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import nb_asr_b200 as nb  # noqa: E402
from gpu_utils import DEV, geo, stream, unpack_mask  # noqa: E402
from nb_asr_b200 import _lib, proxies, sweep  # noqa: E402
from oracle import model_ref as M  # noqa: E402
from oracle import nwot_ref as R  # noqa: E402

ARCHS = {'linear_skips': [[0, 1], [0, 1, 1], [0, 1, 1, 1]], 'c7d2_skips': [[4, 1], [4, 1, 1], [4, 1, 1, 1]],
         'mixed': [[2, 1], [3, 0, 1], [0, 1, 0, 1]], 'zero_mix': [[5, 1], [1, 1, 0], [5, 0, 1, 1]],
         'default': [[1, 0], [1, 0, 0], [1, 0, 0, 0]]}
B, T = 8, 200


def build(arch, precision):
    nb.set_seed(1235)
    return nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision=precision).eval()


def batch():
    return nb.data.make_batch(B, T, seed=0, min_len=T // 2)


def valid_frames(alen, T_k, k):
    return torch.tensor([proxies.gate_frames(int(a), T_k, proxies.LEN_SHIFT[k]) for a in alen], device=DEV)


def ref_gram(layers, alen):
    """torch reference: unpack every layer's bits, drop frames >= L, K = A A^T + B B^T in fp64 (exact integers)."""
    nb_ = len(alen)
    K = torch.zeros(nb_, nb_, dtype=torch.float64, device=DEV)
    for mask, w, Cc, T_k, k in layers:
        m = unpack_mask(mask, nb_, T_k, Cc, w)                                          # (B, T_k, C)
        valid = (torch.arange(T_k, device=DEV)[None, :] < valid_frames(alen, T_k, k)[:, None])[:, :, None]
        a = (m & valid).reshape(nb_, -1).double()
        b = (~m & valid).reshape(nb_, -1).double()
        K += a @ a.T + b @ b.T
    return K.cpu().numpy().astype(np.uint64)


def run_gram(layers, alen):
    """nbasr_gate_gram over [(mask (planes, rows, eb) uint8, w, C, T_k, block k)]; K uint64 numpy.  K starts as garbage."""
    lib = _lib.load()
    nb_ = len(alen)
    arr = (_lib.GateLayer * len(layers))()
    for e, (mask, w, Cc, T_k, k) in zip(arr, layers):
        e.mask, e.mask_rows, e.w, e.C, e.Tp, e.T, e.s = mask.data_ptr(), mask.shape[1], w, Cc, geo(T_k), T_k, proxies.LEN_SHIFT[k]
    table = torch.frombuffer(bytearray(arr), dtype=torch.uint8).to(DEV)
    lens = torch.tensor(alen, dtype=torch.int64, device=DEV)
    K = torch.full((nb_, nb_), -1, dtype=torch.int64, device=DEV)
    work = torch.full((int(lib.nbasr_gate_gram_work_elems(nb_)),), -1, dtype=torch.int64, device=DEV)
    rc = lib.nbasr_gate_gram(table.data_ptr(), len(layers), lens.data_ptr(), nb_, K.data_ptr(), work.data_ptr(), stream())
    torch.cuda.synchronize()
    _lib.check(rc, 'gate_gram')
    return K.cpu().numpy().view(np.uint64)


def random_layers(nb_, T0, seed):
    """every plane width with every channel count, on the four blocks' frame counts; all bytes random: bits beyond C, bits
    >= w of 8-byte entries, pad rows and frames >= L are garbage the kernel must ignore"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    t_blk, tt = [], T0
    for s in (1, 1, 2, 2):
        tt = tt if s == 1 else (tt + 1) // 2
        t_blk.append(tt)
    layers = []
    for n, (w, Cc) in enumerate([(w, c) for w in (32, 40, 48) for c in (600, 800, 1000, 1200)]):
        k = n % 4
        eb = 4 if w == 32 else 8
        rows = nb_ * geo(t_blk[k]) + 8
        mask = torch.randint(0, 256, ((Cc + w - 1) // w, rows, eb), generator=g, device=DEV, dtype=torch.int32).to(torch.uint8)
        layers.append((mask, w, Cc, t_blk[k], k))
    return layers


@pytest.mark.parametrize('nb_', [1, 3, 8, 64, 128])
def test_gate_gram_matches_bit_unpacking_reference(nb_):
    T0 = 70                                                   # 70 / 70 / 35 / 18 frames: several 32-frame chunks
    rng = np.random.default_rng(nb_)
    alen = rng.integers(1, T0 + 1, nb_)
    alen[0] = T0
    if nb_ > 1:
        alen[1] = 1
    if nb_ > 2:
        alen[2] = T0 + 50                                     # longer than the padded batch: capped at T_k
    layers = random_layers(nb_, T0, seed=nb_)
    ref = ref_gram(layers, alen)
    got = run_gram(layers, alen)
    np.testing.assert_array_equal(got, ref)
    np.testing.assert_array_equal(run_gram(layers, alen), got)          # bit-identical on a second call
    assert np.array_equal(got, got.T)


def test_gate_gram_rejects_more_than_128_rows():
    lib = _lib.load()
    layers = random_layers(129, 9, seed=0)
    arr = (_lib.GateLayer * 1)()
    mask, w, Cc, T_k, k = layers[0]
    arr[0].mask, arr[0].mask_rows, arr[0].w, arr[0].C, arr[0].Tp, arr[0].T, arr[0].s = mask.data_ptr(), mask.shape[1], w, Cc, geo(T_k), T_k, 0
    table = torch.frombuffer(bytearray(arr), dtype=torch.uint8).to(DEV)
    lens = torch.full((129,), 9, dtype=torch.int64, device=DEV)
    K = torch.empty(129, 129, dtype=torch.int64, device=DEV)
    work = torch.empty(int(lib.nbasr_gate_gram_work_elems(128)), dtype=torch.int64, device=DEV)
    assert lib.nbasr_gate_gram(table.data_ptr(), 1, lens.data_ptr(), 129, K.data_ptr(), work.data_ptr(), stream()) != 0
    assert b'128' in lib.nbasr_last_error()


# ----------------------------------------------------------------------------------------------- plan masks
def plan_layers(pl):
    out = []
    for mask, g, k in pl.gates:
        eb = 4 if mask.w == 32 else 8
        out.append((mask.t.view((g.C + mask.w - 1) // mask.w, g.rows, eb), mask.w, g.C, g.T, k))
    return out


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('name', list(ARCHS))
def test_plan_masks_kernel_matches_reference(name, precision):
    model = build(ARCHS[name], precision)
    (audio, alen), tgt = batch()
    K = proxies.nwot_kernel(model, ((audio, alen), tgt))
    pl = model.engine.plan(B, T, False, True)
    arch = M.arch_vec_to_names(ARCHS[name])
    n_relu = sum(1 for nd in arch if nd[0] != 'zero')
    assert len(pl.gates) == 4 + sum(M.CELLS) * n_relu
    # plane widths: 32 (GEMM / SIMT producers), 48 / 40 (C = 1000) from the tcgen05 grouped conv of the 16-bit mode
    conv = precision == 'bf16' and any(nd[0] in M.CONV_EDGE for nd in arch)
    assert {m.w for m, _, _ in pl.gates} == ({32, 40, 48} if conv else {32})
    np.testing.assert_array_equal(K, ref_gram(plan_layers(pl), alen.numpy()))


# ----------------------------------------------------------------------------------------------- oracle
_ORACLE = {}


def oracle_codes(name):
    if name not in _ORACLE:
        (audio, alen), _ = batch()
        _ORACLE[name] = R.gate_codes(M.build_state_dict(ARCHS[name], seed=1235), ARCHS[name], audio)
    return _ORACLE[name]


def disagreements(pl, codes, alen):
    """per utterance: number of valid units whose engine code differs from the oracle's"""
    d = np.zeros(B, np.int64)
    assert len(pl.gates) == len(codes)
    for (mask, w, Cc, T_k, k), (k2, m_ref) in zip(plan_layers(pl), codes):
        assert k == k2 and m_ref.shape == (B, Cc, T_k)
        m = unpack_mask(mask, B, T_k, Cc, w).permute(0, 2, 1).cpu()
        valid = torch.arange(T_k)[None, :] < torch.as_tensor(R.frames(alen, T_k, k))[:, None]
        d += ((m != m_ref) & valid[:, None, :]).sum((1, 2)).numpy()
    return d


# 16-bit mode: fp16 activations move pre-activations that sit within rounding of 0 or 20 across the gate.  Measured on a
# B200 (1 000 W, this fixture), largest fraction of an utterance's valid units whose code differs from the fp64 oracle:
# 5.7e-4 (linear_skips), 4.2e-4 (c7d2_skips), 4.7e-4 (mixed), 3.7e-4 (zero_mix); largest K error 5.9e-5 of K_ii; relative
# score error <= 4.3e-7 (fp32 mode: disagreement <= 4.2e-6, K error <= 3.5e-6 of K_ii, score <= 1.1e-7).  The bounds
# below keep 3.5x / 20x headroom over those (DESIGN.md 7b); K itself is also held to the exact bound the measured
# disagreements give.  The default arch is not compared in 16-bit mode: at the reference initialisation its activations
# vanish with depth and fp16 flushes them (DESIGN.md 4).
BF16_GATE_FRAC = 2e-3
BF16_SCORE_TOL = 1e-5


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('name', list(ARCHS))
def test_nwot_matches_oracle(name, precision):
    if precision == 'bf16' and name == 'default':
        pytest.skip('default arch at reference init: fp16 flushes its vanishing activations (DESIGN.md 4)')
    (audio, alen), tgt = batch()
    codes = oracle_codes(name)
    K_ref = R.kernel_from_codes(codes, alen.numpy())
    s_ref = R.nwot_score(K_ref)
    model = build(ARCHS[name], precision)
    K = proxies.nwot_kernel(model, ((audio, alen), tgt)).astype(np.float64)
    pl = model.engine.plan(B, T, False, True)
    d = disagreements(pl, codes, alen.numpy())
    diag = np.diag(K_ref)
    err = np.abs(K - K_ref)
    # flipping one unit of utterance i changes K[i, j] by at most one: the error is bounded by the disagreement counts
    assert np.all(err <= d[:, None] + d[None, :])
    s = proxies.nwot_score(K)
    frac = float((d / diag).max())
    print(f'nwot {name}/{precision}: gate disagreement max {frac:.3e}, K err max {float((err / diag[:, None]).max()):.3e} '
          f'of K_ii, score {s:.6f} ref {s_ref:.6f} rel {abs(s - s_ref) / abs(s_ref):.3e}', file=sys.stderr)
    assert np.isfinite(s_ref)
    if precision == 'fp32':
        assert np.all(err <= 1e-4 * diag[:, None]), (err / diag[:, None]).max()
        assert abs(s - s_ref) <= 1e-3 * abs(s_ref), (s, s_ref)
    else:
        assert frac <= BF16_GATE_FRAC, frac
        assert abs(s - s_ref) <= BF16_SCORE_TOL * abs(s_ref), (s, s_ref)


# ----------------------------------------------------------------------------------------------- compute_proxies / sweep
OTHERS = ('grad_norm', 'snip', 'synflow', 'jacob_cov')


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_compute_proxies_nwot_alone_equals_shared(precision):
    model = build(ARCHS['mixed'], precision)
    b = batch()
    alone = proxies.compute_proxies(model, b, ('nwot',))
    shared = proxies.compute_proxies(model, b, ('grad_norm', 'snip', 'nwot'))
    every = proxies.compute_proxies(model, b)
    assert np.isfinite(alone['nwot'])
    assert alone['nwot'] == shared['nwot'] == every['nwot']
    assert alone['nwot'] == proxies.nwot_score(proxies.nwot_kernel(model, b))
    before = proxies.compute_proxies(model, b, OTHERS)
    for m in OTHERS:                       # fp32 atomics of the weight-gradient kernels, as in test_gpu_10
        assert every[m] == pytest.approx(before[m], rel=1e-5), (m, every[m], before[m])
    assert proxies.compute_proxies(model, b, ('nwot',), per_layer=True)['nwot'] == alone['nwot']


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_nwot_leaves_the_model_state_untouched(precision):
    model = build(ARCHS['zero_mix'], precision)
    tr = nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[0], verbose=False)
    tr.model = tr._model = model
    tr.optimizer = nb.trainer.FusedAdam(model, lr=1e-4)
    model.train()
    tr.step(batch(), training=True)
    model.eval()
    eng = model.engine
    before = [t.clone() for t in (eng.flat_p, eng.flat_g, eng.adam_m, eng.adam_v, eng.opt_state, eng.drop_step)]
    with torch.no_grad():
        l0 = model(batch()[0][0].to(DEV))
    proxies.compute_proxies(model, batch(), ('nwot',))
    with torch.no_grad():
        l1 = model(batch()[0][0].to(DEV))
    for a, b_ in zip(before, (eng.flat_p, eng.flat_g, eng.adam_m, eng.adam_v, eng.opt_state, eng.drop_step)):
        assert torch.equal(a, b_)
    assert torch.equal(l0, l1)


def test_duplicated_utterance_scores_minus_inf():
    model = build(ARCHS['mixed'], 'bf16')
    (audio, alen), (tg, tl) = batch()
    audio[3], alen[3] = audio[1], alen[1]
    K = proxies.nwot_kernel(model, ((audio, alen), (tg, tl)))
    assert np.array_equal(K[3], K[1]) and K[1, 3] == K[1, 1]
    assert proxies.compute_proxies(model, ((audio, alen), (tg, tl)), ('nwot',))['nwot'] == -np.inf


def test_sweep_nwot_column(tmp_path, monkeypatch):
    import pickle
    arch = ARCHS['zero_mix']
    batches = [nb.data.make_batch(B, T, seed=100 + i, min_len=T // 3) for i in range(2)]
    batches = [((a.to(DEV), al.to(DEV)), (t.to(DEV), tl.to(DEV))) for (a, al), (t, tl) in batches]
    gain = 101 ** 0.5
    row = sweep.evaluate_arch(arch, batches, 0, 'bf16', seed=7, init='device', conv_gain=gain, proxies=('nwot',))
    model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision='bf16', init='device', seed=7, conv_gain=gain)
    model.eval()
    direct = proxies.compute_proxies(model, batches[0], ('nwot',))['nwot']
    assert np.isfinite(row['nwot']) and row['nwot'] == direct
    out = tmp_path / 'rows.pkl'
    monkeypatch.setattr(sys, 'argv', ['sweep', '--limit', '1', '--dataset', 'uniform', '--batch', '8', '--frames', '120',
                                      '--n-batches', '1', '--proxies', 'nwot', '--out-pickle', str(out)])
    sweep.main()
    with open(out, 'rb') as f:
        header, rows = pickle.load(f), pickle.load(f)
    assert header['columns'][-1] == 'nwot' and header['proxy_batches'] == 1
    assert len(rows) == 1 and np.isfinite(rows[0][-1])
