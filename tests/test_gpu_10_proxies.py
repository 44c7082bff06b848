"""-m gpu: input gradients through the engine and the zero-cost proxies (nb_asr_b200.proxies) -- the three proxy kernels
against torch fp64, the N = 80 input-gradient GEMM, audio.grad and every proxy against the fp64 CPU oracle
(oracle/proxies_ref.py), and the state a proxy call must leave untouched.  Small fixture sizes (B = 8, T = 200): the fp64
oracle runs on the CPU."""

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import nb_asr_b200 as nb  # noqa: E402
from gpu_utils import DEV, epilogue, geo, relerr, run_gemm, stream  # noqa: E402
from nb_asr_b200 import _lib, proxies, sweep  # noqa: E402
from nb_asr_b200._lib import BF16, F32, PAD_L  # noqa: E402
from oracle import model_ref as M  # noqa: E402
from oracle import proxies_ref as R  # noqa: E402

ARCHS = {'linear_skips': [[0, 1], [0, 1, 1], [0, 1, 1, 1]], 'c7d2_skips': [[4, 1], [4, 1, 1], [4, 1, 1, 1]],
         'mixed': [[2, 1], [3, 0, 1], [0, 1, 0, 1]], 'zero_mix': [[5, 1], [1, 1, 0], [5, 0, 1, 1]]}
B, T = 8, 200
# whole-model gradient bounds of test_gpu_5_model.py (per tensor 2e-2, cosine > 1 - 1e-4)
GRAD_TOL = 2e-2


def build(arch, precision):
    nb.set_seed(1235)
    return nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision=precision).eval()


def batch():
    return nb.data.make_batch(B, T, seed=0, min_len=T // 2)


def cosine(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float(a @ b / (a.norm() * b.norm()))


# ----------------------------------------------------------------------------------------------- kernels
def test_param_stats_matches_fp64_and_is_deterministic():
    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    lens = [1, 17, 16383, 16384, 16385, 40001, 3, 100003]
    offs, o = [], 0
    for i, n in enumerate(lens):
        o += 5 if i % 2 else 64           # odd offsets take the scalar path
        offs.append(o)
        o += n
    p = (torch.randn(o, generator=g) * 0.05).to(DEV)
    gr = (torch.randn(o, generator=g) * 1e-20).to(DEV)          # squares of ~1e-20 underflow fp32
    off = torch.tensor(offs, dtype=torch.int64, device=DEV)
    ln = torch.tensor(lens, dtype=torch.int64, device=DEV)
    chunks = sum((n + 16383) // 16384 for n in lens)
    part = torch.empty(2 * chunks, dtype=torch.float64, device=DEV)
    res = []
    for _ in range(2):
        out = torch.full((len(lens), 2), float('nan'), dtype=torch.float64, device=DEV)
        _lib.check(lib.nbasr_param_stats(p.data_ptr(), gr.data_ptr(), off.data_ptr(), ln.data_ptr(), len(lens), chunks,
                                         part.data_ptr(), out.data_ptr(), stream()), 'param_stats')
        torch.cuda.synchronize()
        res.append(out.cpu())
    assert torch.equal(res[0], res[1])
    p64, g64 = p.double().cpu(), gr.double().cpu()
    for s, (a, n) in enumerate(zip(offs, lens)):
        sq = float((g64[a:a + n] ** 2).sum())
        ab = float((p64[a:a + n] * g64[a:a + n]).abs().sum())
        assert sq > 0 and abs(res[0][s, 0].item() - sq) <= 1e-12 * sq, (s, res[0][s, 0].item(), sq)
        assert abs(res[0][s, 1].item() - ab) <= 1e-12 * ab, (s, res[0][s, 1].item(), ab)


@pytest.mark.parametrize('b,D,ld', [(8, 10007, 10240), (64, 41 * 80, 41 * 80), (3, 5, 5)])
def test_row_gram_matches_fp64(b, D, ld):
    lib = _lib.load()
    x = torch.randn(b, ld, generator=torch.Generator().manual_seed(b)) + 0.3
    xd = x.to(DEV)
    gram = torch.empty(b, b, dtype=torch.float64, device=DEV)
    rs = torch.empty(b, dtype=torch.float64, device=DEV)
    work = torch.empty(((D + 255) // 256) * (b * (b + 1) // 2 + b), dtype=torch.float64, device=DEV)
    got = []
    for _ in range(2):
        _lib.check(lib.nbasr_row_gram(xd.data_ptr(), b, D, ld, gram.data_ptr(), rs.data_ptr(), work.data_ptr(), stream()), 'row_gram')
        torch.cuda.synchronize()
        got.append((gram.cpu().clone(), rs.cpu().clone()))
    assert torch.equal(got[0][0], got[1][0]) and torch.equal(got[0][1], got[1][1])
    x64 = x[:, :D].double()
    torch.testing.assert_close(got[0][0], x64 @ x64.T, rtol=1e-12, atol=1e-9)
    torch.testing.assert_close(got[0][1], x64.sum(1), rtol=1e-12, atol=1e-9)


def test_transpose_out_matches_permute():
    lib = _lib.load()
    b, F, t = 3, 80, 77
    Tp = geo(t)
    src = torch.randn(b * Tp + 8, F, device=DEV)
    out = torch.full((b, F, t), float('nan'), device=DEV)
    _lib.check(lib.nbasr_transpose_out(src.data_ptr(), out.data_ptr(), b, F, t, Tp, stream()), 'transpose_out')
    torch.cuda.synchronize()
    ref = src[:b * Tp].view(b, Tp, F)[:, PAD_L:PAD_L + t].permute(0, 2, 1)
    assert torch.equal(out, ref)


@pytest.mark.parametrize('dt', [BF16, F32])
def test_input_gradient_gemm_n80(dt):
    """Block 0's input-gradient GEMM: K = 8 * 600 over overlapping rows of the padded dZ, N = 80 (not a multiple of the
    pair kernel's 64-row W half-tiles: TMA zero-fills rows 80..127, the direct fp32 epilogue masks columns >= 80)."""
    b, t, Cc, N = 3, 150, 600, 80
    Tp = geo(t)
    tdt = torch.bfloat16 if dt == BF16 else torch.float32
    g = torch.Generator().manual_seed(1)
    dz = torch.zeros(b * Tp + 8, Cc)
    dz[:b * Tp].view(b, Tp, Cc)[:, PAD_L:PAD_L + t] = torch.randn(b, t, Cc, generator=g)
    w = torch.randn(N, 8 * Cc, generator=g) * 0.02
    dz_d, w_d = dz.to(DEV, tdt), w.to(DEV, tdt)
    out = torch.zeros(b * Tp + 8, N, device=DEV)
    epi = epilogue(dt, N, out=out, out_dtype=F32)
    run_gemm(dt, dz_d.data_ptr() + (PAD_L - 4) * Cc * dz_d.element_size(), Tp * Cc, Cc, b, t, 8 * Cc, N, w_d, 8 * Cc, PAD_L, Tp, 1, epi)
    dz64, w64 = dz_d.double().cpu(), w_d.double().cpu()
    z3 = dz64[:b * Tp].view(b, Tp, Cc)
    A = torch.cat([z3[:, PAD_L - 4 + q:PAD_L - 4 + q + t] for q in range(8)], dim=2)      # (b, t, 8 * Cc)
    ref = A @ w64.T
    got = out[:b * Tp].view(b, Tp, N).double().cpu()
    assert relerr(got[:, PAD_L:PAD_L + t], ref) < 1e-5
    assert not got[:, :PAD_L].any() and not got[:, PAD_L + t:].any()
    assert not out[b * Tp:].any()


# ----------------------------------------------------------------------------------------------- input gradients
W0 = 'model.0.conv.weight'


def ref_input_grads(arch, audio, alen, tg, tl):
    """fp64 oracle: (input gradient, conv_0 weight gradient) of sum(logits) and of the CTC loss"""
    sd = {k: v.double().requires_grad_(True) for k, v in M.build_state_dict(arch, seed=1235).items()}
    out = []
    for f in (lambda y: y.sum(), lambda y: M.ctc_loss_ref(torch.log_softmax(y, 2), alen // 4, tg, tl)):
        sd[W0].grad = None
        x = audio.double().clone().requires_grad_(True)
        f(M.forward(sd, arch, x)).backward()
        out.append((x.grad.clone(), sd[W0].grad.clone()))
    return out


# 16-bit mode: the input gradient is block 0's bf16 dZ times W, and conv_0's weight gradient is the same dZ against the
# input, so both carry the error of the bf16 backward pass down to block 0 (fp16 activations and bf16 gradients through
# ~80 layers).  Measured on a B200 (B = 8, T = 200, CTC loss), input-gradient / conv_0 weight-gradient error against the
# fp64 oracle: linear_skips 0.102 / 0.102, c7d2_skips 0.051 / 0.051, mixed 0.074 / 0.074, zero_mix 0.049 / 0.049; the
# fp32 engine's input gradient differs from the 16-bit one by the same amount.  So the 16-bit input gradient is held to
# the accuracy of the existing weight gradient it shares its dZ with (ratio <= 1.5) and to a cosine bound; the fp32 mode
# pins the path itself with the whole-model bounds of test_gpu_5_model.py.
BF16_INPUT_GRAD_RATIO = 1.5
BF16_INPUT_GRAD_COS = 0.99


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('name', ['linear_skips', 'c7d2_skips'])
def test_audio_grad_matches_oracle(name, precision):
    arch = ARCHS[name]
    (audio, alen), (tg, tl) = batch()
    (g_sum, w_sum), (g_loss, w_loss) = ref_input_grads(arch, audio, alen, tg, tl)
    model = build(arch, precision)
    w0 = dict(model.named_parameters())[W0]

    def check(xg, g_ref, w_ref):
        e, c = relerr(xg.cpu(), g_ref), cosine(xg, g_ref)
        if precision == 'fp32':
            assert e < GRAD_TOL and c > 1 - 1e-4, (e, c)
        else:
            ew = relerr(w0.grad.cpu(), w_ref)
            assert e <= BF16_INPUT_GRAD_RATIO * ew and c > BF16_INPUT_GRAD_COS, (e, ew, c)

    x = audio.to(DEV).requires_grad_(True)
    model(x).sum().backward()
    assert x.grad is not None and x.grad.shape == x.shape and x.grad.dtype == torch.float32
    check(x.grad, g_sum, w_sum)
    first = x.grad.clone()
    model(x).sum().backward()                       # accumulates like autograd
    torch.testing.assert_close(x.grad, 2 * first, rtol=1e-6, atol=0)
    for p in model.parameters():
        p.grad.zero_()
    x = audio.to(DEV).requires_grad_(True)
    logp = torch.log_softmax(model(x), 2)
    nb.get_loss()(logp, (alen // 4).to(DEV), tg.to(DEV), tl.to(DEV)).backward()
    check(x.grad, g_loss, w_loss)


def test_input_gradient_plan_appends_three_calls_and_keeps_the_others():
    model = build(ARCHS['mixed'], 'bf16')
    eng = model.engine
    plain = eng.plan(B, T, False, True)
    withx = eng.plan(B, T, False, True, input_grad=True)
    assert (B, T, False, True) in eng.plans and (B, T, False, True, 'input_grad') in eng.plans
    assert plain.daudio is None
    names = lambda ops: [fn.__name__ for fn, _ in ops]               # noqa: E731
    assert names(withx.fwd) == names(plain.fwd)
    assert names(withx.bwd) == names(plain.bwd) + ['nbasr_pack_weight', 'nbasr_gemm_tn', 'nbasr_transpose_out']
    assert withx.buckets == plain.buckets
    # the engine-wide pack table (refreshed by every optimiser step) does not grow
    assert eng.pack_njobs == len(eng.pack_ops) and 'model.0.conv' not in eng.wd


# ----------------------------------------------------------------------------------------------- proxies
_ORACLE = {}


def oracle(name):
    if name not in _ORACLE:
        arch = ARCHS[name]
        sd = M.build_state_dict(arch, seed=1235)
        (audio, alen), (tg, tl) = batch()
        corr, _ = R.jacob_corr(sd, arch, audio)
        _ORACLE[name] = dict(gs=R.grad_stats(sd, arch, audio, alen, tg, tl), corr=corr, jc=R.jacob_cov_score(corr),
                             sf=R.synflow(sd, arch, T))
    return _ORACLE[name]


# Relative bounds on the totals: fp32 mode 1e-3, 16-bit mode 2e-2; jacob_cov on the correlation matrix (max abs entry
# difference), its score only in fp32 mode.
TOTAL_TOL = {'fp32': 1e-3, 'bf16': 2e-2}
CORR_TOL = {'fp32': 1e-3, 'bf16': 2e-2}


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
@pytest.mark.parametrize('name', list(ARCHS))
def test_proxies_match_oracle(name, precision):
    ref = oracle(name)
    model = build(ARCHS[name], precision)
    got = proxies.compute_proxies(model, batch(), per_layer=True)
    tol = TOTAL_TOL[precision]
    gn_ref = sum(v[0] for v in ref['gs'].values())
    sn_ref = sum(v[1] for v in ref['gs'].values())
    assert set(got['grad_norm']) == set(ref['gs']) == set(got['snip'])
    gn, sn = sum(got['grad_norm'].values()), sum(got['snip'].values())
    assert abs(gn - gn_ref) <= tol * gn_ref, (gn, gn_ref)
    assert abs(sn - sn_ref) <= tol * sn_ref, (sn, sn_ref)
    # synflow always runs on the fp32 norm-free copy
    sf, sf_ref = sum(got['synflow'].values()), sum(ref['sf'].values())
    assert abs(sf - sf_ref) <= 1e-3 * sf_ref, (sf, sf_ref)
    corr = proxies.jacob_correlation(model, batch()[0][0].to(DEV))
    err = float(np.abs(corr - ref['corr']).max())
    assert err < CORR_TOL[precision], err
    if precision == 'fp32':
        assert abs(got['jacob_cov'] - ref['jc']) <= 1e-3 * abs(ref['jc']), (got['jacob_cov'], ref['jc'])
    # the weight-gradient kernels accumulate with fp32 atomics: a second backward pass agrees to fp32 rounding only
    totals = proxies.compute_proxies(model, batch())
    assert totals['grad_norm'] == pytest.approx(gn, rel=1e-5) and totals['synflow'] == pytest.approx(sf, rel=1e-5)


def test_prunable_copy_forward_matches_oracle_without_norm():
    arch = ARCHS['mixed']
    model = build(arch, 'fp32')
    cp = model.get_prunable_copy(bn=False).set_precision('fp32').eval()
    (audio, _), _ = batch()
    with torch.no_grad():
        got = cp(audio.to(DEV))
    ref = M.forward(M.build_state_dict(arch, seed=1235), arch, audio, use_norm=False)
    assert relerr(got.cpu(), ref) < 1e-4, relerr(got.cpu(), ref)
    fast = proxies._norm_free_fp32_copy(model)
    assert torch.equal(fast.engine.flat_p, cp.engine.flat_p)


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_proxies_leave_the_model_state_untouched(precision):
    model = build(ARCHS['zero_mix'], precision)
    tr = nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[0], verbose=False)
    tr.model = tr._model = model
    tr.optimizer = nb.trainer.FusedAdam(model, lr=1e-4)
    model.train()
    tr.step(batch(), training=True)                  # non-trivial Adam state and gradients
    model.eval()
    eng = model.engine
    before = [t.clone() for t in (eng.flat_p, eng.flat_g, eng.adam_m, eng.adam_v, eng.opt_state, eng.drop_step)]
    with torch.no_grad():
        l0 = model(batch()[0][0].to(DEV))
    proxies.compute_proxies(model, batch())
    # synflow on the model itself (norm-free fp32 copies only: here the signs of its own parameters are flipped)
    cp = proxies._norm_free_fp32_copy(model)
    p_cp = cp.engine.flat_p.clone()
    with torch.no_grad():
        c0 = cp(batch()[0][0].to(DEV))
    proxies.synflow_stats(model, T, copy=cp)
    assert torch.equal(cp.engine.flat_p, p_cp)
    with torch.no_grad():
        assert torch.equal(cp(batch()[0][0].to(DEV)), c0)
        l1 = model(batch()[0][0].to(DEV))
    after = (eng.flat_p, eng.flat_g, eng.adam_m, eng.adam_v, eng.opt_state, eng.drop_step)
    for a, b_ in zip(before, after):
        assert torch.equal(a, b_)
    assert torch.equal(l0, l1)


def test_sweep_row_equals_compute_proxies():
    arch = ARCHS['zero_mix']
    batches = [nb.data.make_batch(B, T, seed=100 + i, min_len=T // 3) for i in range(2)]
    batches = [((a.to(DEV), al.to(DEV)), (t.to(DEV), tl.to(DEV))) for (a, al), (t, tl) in batches]
    gain = 101 ** 0.5
    row = sweep.evaluate_arch(arch, batches, 0, 'bf16', seed=7, init='device', conv_gain=gain, proxies=proxies.MEASURES,
                              proxy_batches=2)
    plain = sweep.evaluate_arch(arch, batches, 0, 'bf16', seed=7, init='device', conv_gain=gain)
    assert set(row) == set(plain) | set(proxies.MEASURES)
    assert all(row[k] == plain[k] for k in plain)
    model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision='bf16', init='device', seed=7, conv_gain=gain)
    model.eval()
    direct = [proxies.compute_proxies(model, b) for b in batches]     # (same values up to the fp32 atomics of the backward)
    for m in proxies.MEASURES:
        v = sum(d[m] for d in direct) / 2
        assert np.isfinite(row[m]) and row[m] == pytest.approx(v, rel=1e-5, abs=0), (m, row[m], v)
