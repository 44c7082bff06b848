"""-m gpu: parity of the paths bench.py actually times -- CUDA-graph replay of the step, the bucketed NCCL
data-parallel step -- plus the 16-bit mode at the sizes BASELINE.json quotes (cfg 2: 64 x 500, cfg 5: 32 x 3000 mixed).

Reference semantics matched: training/torch/trainer.py:208-227 (step), :36-44 (loss), :91-92 (DataParallel)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import nb_asr_b200 as nb  # noqa: E402
from conftest import ROOT, golden_path  # noqa: E402
from oracle import decode_np as D  # noqa: E402
from oracle import model_ref as M  # noqa: E402

DEV = 'cuda:0'
LOGIT_TOL_16 = 2e-2          # north_star: logits and CTC loss within 2e-2 relative in the 16-bit mode


def rel64(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm())


def make(arch, precision, graph, dropout=0.0, lr=1e-4):
    nb.set_seed(1235)
    model = nb.get_model(arch, use_rnn=True, dropout_rate=dropout, gpu=0, precision=precision)
    tr = nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[0], save_dir=None, verbose=False)
    tr.model = tr._model = model
    tr.optimizer = nb.trainer.FusedAdam(model, lr=lr)
    tr.use_graph = graph
    return model, tr


@pytest.mark.parametrize('name', ['c7d2_skips', 'mixed'])
def test_graph_train_steps_match_reference_and_eager_fp32(name, golden_meta):
    """use_graph=True (what bench.py times): two consecutive fp32 train steps against the REAL reference's Trainer.step
    (tests/golden/meta.json loss0 / params0 / loss1) and against the eager path, with an lr change between the steps."""
    meta = golden_meta[f'train_{name}']
    batch = nb.data.make_batch(meta['B'], meta['T'], seed=0, min_len=meta['T'] // 2)
    res = {}
    for graph in (False, True):
        model, tr = make(meta['arch'], 'fp32', graph)
        model.train()
        l0, lp0, _ = tr.step(batch, training=True)
        p0 = model.engine.flat_p.clone()
        l1, lp1, _ = tr.step(batch, training=True)
        tr.optimizer.param_groups[0]['lr'] = 5e-5            # lr lives on the device; the graph must pick the change up
        l2, _, _ = tr.step(batch, training=True)
        res[graph] = (l0.item(), lp0.clone(), p0, l1.item(), lp1.clone(), model.engine.flat_p.clone(), l2.item(), model)
    e, g = res[False], res[True]
    assert tr.use_graph, 'graph capture fell back to eager'
    # forward pass is deterministic: the first step's loss and log-probs are BIT-equal between graph replay and eager
    assert g[0] == e[0] and torch.equal(g[1], e[1])
    # after the update only the order of the fp32 atomic weight-gradient sums differs (Adam turns a sign flip of a ~0
    # gradient element into a +-lr step: a few 1e-6 of the parameter norm)
    assert rel64(g[2], e[2]) < 1e-5 and abs(g[3] - e[3]) < 1e-4 * abs(e[3]) and rel64(g[4], e[4]) < 1e-4
    assert rel64(g[5], e[5]) < 2e-5 and abs(g[6] - e[6]) < 1e-4 * abs(e[6])
    # ... and the graph path against the real reference
    assert abs(g[0] - meta['loss0']) < 1e-4 * abs(meta['loss0'])
    assert abs(g[3] - meta['loss1']) < 2e-3 * abs(meta['loss1'])
    model = g[7]
    # params0 of the golden file = parameters after the FIRST reference step: rebuild and compare after one graph step
    model1, tr1 = make(meta['arch'], 'fp32', True)
    model1.train()
    tr1.step(batch, training=True)
    sd = model1.state_dict()
    for k, s in meta['params0'].items():
        v = sd[k].double().cpu()
        assert abs(float(v.sum()) - s['sum']) <= 2e-4 * abs(s['sum']) + 2e-3, k
        assert np.allclose(v.flatten()[:8].numpy(), s['head'], rtol=2e-4, atol=2e-6), k


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_graph_eval_and_dropout_steps_are_bit_equal_to_eager(precision):
    """Eval step (fwd + CTC + greedy PER): graph replay == eager, bit for bit; with dropout > 0 the in-graph step counter
    must give the same masks as the eager path (capture warm-up is rolled back)."""
    arch = [[2, 1], [3, 0, 1], [0, 1, 0, 1]]
    batch = nb.data.make_batch(4, 150, seed=2, min_len=90)
    out = {}
    for graph in (False, True):
        model, tr = make(arch, precision, graph, dropout=0.2)
        model.eval()
        le, lpe, ol = tr.step(batch, training=False)
        le2, lpe2, _ = tr.step(batch, training=False)        # second replay of the same graph
        per = tr.decode(lpe, ol, batch)
        model.train()
        lt, lpt, _ = tr.step(batch, training=True)           # dropout active: masks from (seed, in-graph step counter)
        lt2, lpt2, _ = tr.step(batch, training=True)
        out[graph] = (le.item(), lpe.clone(), per.item(), lt.item(), lpt.clone(), lt2.item(), le2.item(), lpe2.clone())
        assert tr.use_graph == graph
    e, g = out[False], out[True]
    assert g[0] == e[0] and torch.equal(g[1], e[1]) and g[2] == e[2]
    assert g[6] == e[6] and torch.equal(g[7], e[7]) and g[6] == g[0]
    assert g[3] == e[3] and torch.equal(g[4], e[4])           # same dropout masks on the first training step
    assert torch.isfinite(torch.tensor(g[5])) and abs(g[5] - e[5]) < 1e-3 * abs(e[5])
    assert not torch.equal(g[4], g[1])                        # dropout really was active


def _label_stats(logp_ours, logp_ref, out_len, tg, tl):
    """Greedy decode of both log-prob tensors through the numpy oracle: frame-level argmax agreement, number of
    utterances whose folded label sequence differs, PERs."""
    per_o, d_o, _, h_o = D.per_batch(logp_ours, out_len, tg, tl)
    per_r, d_r, _, h_r = D.per_batch(logp_ref, out_len, tg, tl)
    agree = n = 0
    for b in range(logp_ours.shape[0]):
        L = int(out_len[b])
        agree += int((logp_ours[b, :L].argmax(-1) == logp_ref[b, :L].argmax(-1)).sum())
        n += L
    mism = sum(1 for a, b in zip(h_o, h_r) if list(a) != list(b))
    return agree / max(n, 1), mism, per_o, per_r


def test_16bit_cfg2_batch_64x500_against_oracle():
    """cfg 2 shape (64 x 500 x 80).  Skip-connected arch: logits within 2e-2, loss within 2e-2, PER kernel bit-exact on our
    log-probs, end-to-end label agreement with the fp32 oracle reported.  Default (skip-free) arch: its activations vanish
    at reference init (SURVEY finding 5: logits ~1e-25), so only loss and the all-blank decode are meaningful."""
    B, T = 64, 500
    batch = nb.data.make_batch(B, T, seed=0, min_len=T, tgt_lo=20, tgt_hi=50)
    (audio, alen), (tg, tl) = batch
    for name, arch in (('c7d2_skips', [[4, 1], [4, 1, 1], [4, 1, 1, 1]]), ('default', [[1, 0], [1, 0, 0], [1, 0, 0, 0]])):
        sd = M.build_state_dict(arch, seed=1235)
        with torch.no_grad():
            ref_loss, ref_logp, out_len, ref_logits = M.eval_step(sd, arch, audio, alen, tg, tl)
        model, tr = make(arch, 'bf16', True)
        model.eval()
        loss, logp, ol = tr.step(batch, training=False)
        per = tr.decode(logp, ol, batch)
        assert ol.cpu().tolist() == out_len.tolist()
        assert abs(loss.item() - ref_loss.item()) < LOGIT_TOL_16 * abs(ref_loss.item())
        rper, rd, _, _ = D.per_batch(logp.cpu().numpy(), ol.cpu().numpy(), tg.numpy(), tl.numpy())
        assert per.item() == rper and tr.last_hyp[2].cpu().tolist() == rd.tolist()          # PER bit-exact
        agree, mism, per_o, per_r = _label_stats(logp.cpu().numpy(), ref_logp.numpy(), out_len.numpy(), tg.numpy(), tl.numpy())
        if name == 'default':
            assert per_o == per_r == 1.0 and mism == 0          # all-blank decode on both sides
        else:
            with torch.no_grad():
                logits = model(audio.to(DEV))
            r = rel64(logits, ref_logits)
            print(f'cfg2 {name}: logits rel {r:.3e}, loss {loss.item():.6f} vs {ref_loss.item():.6f}, argmax agreement '
                  f'{agree:.4f}, utterances with a different label sequence {mism}/{B}, PER {per_o:.4f} vs {per_r:.4f}')
            assert r < LOGIT_TOL_16, r
            assert agree > 0.9
            assert abs(per_o - per_r) < 0.05 * per_r


def test_16bit_cfg5_long_mixed_lengths_against_oracle():
    """cfg 5 shape: 32 x 3000 frames, mixed lengths (zero padded), one infeasible alignment (zero_infinity)."""
    B, T = 32, 3000
    arch = [[3, 1], [0, 0, 1], [2, 1, 0, 0]]
    (audio, alen), (tg, tl) = nb.data.make_batch(B, T, seed=5, min_len=750, tgt_lo=60, tgt_hi=180)
    alen[3] = 4 * 30                       # 30 output frames for >= 60 labels: infeasible -> zero loss / zero gradient
    audio[3, :, 120:] = 0.0
    batch = ((audio, alen), (tg, tl))
    sd = M.build_state_dict(arch, seed=1235)
    with torch.no_grad():
        ref_loss, ref_logp, out_len, ref_logits = M.eval_step(sd, arch, audio, alen, tg, tl)
    model, tr = make(arch, 'bf16', True)
    model.eval()
    loss, logp, ol = tr.step(batch, training=False)
    per = tr.decode(logp, ol, batch)
    with torch.no_grad():
        logits = model(audio.to(DEV))
    assert logits.shape == (B, 750, 49)
    r = rel64(logits, ref_logits)
    agree, mism, per_o, per_r = _label_stats(logp.cpu().numpy(), ref_logp.numpy(), out_len.numpy(), tg.numpy(), tl.numpy())
    print(f'cfg5: logits rel {r:.3e}, loss {loss.item():.6f} vs {ref_loss.item():.6f}, argmax agreement {agree:.4f}, '
          f'label sequences differing {mism}/{B}, PER {per_o:.4f} vs {per_r:.4f}')
    assert r < LOGIT_TOL_16, r
    assert abs(loss.item() - ref_loss.item()) < LOGIT_TOL_16 * abs(ref_loss.item())
    rper, rd, _, _ = D.per_batch(logp.cpu().numpy(), ol.cpu().numpy(), tg.numpy(), tl.numpy())
    assert per.item() == rper and tr.last_hyp[2].cpu().tolist() == rd.tolist()
    assert agree > 0.9
    # a training step at this size runs and the infeasible utterance contributes nothing
    model.train()
    l0, _, _ = tr.step(batch, training=True)
    assert torch.isfinite(l0) and abs(l0.item() - ref_loss.item()) < LOGIT_TOL_16 * abs(ref_loss.item())


def test_plan_cache_is_bounded():
    """Loaders whose padded length changes every batch must not accumulate plans (ADVICE r1): LRU of max_plans."""
    model, tr = make([[5, 1], [1, 1, 0], [5, 0, 1, 1]], 'bf16', True)
    model.engine.max_plans = 3
    model.eval()
    for T in (64, 72, 80, 88, 96, 64):
        batch = nb.data.make_batch(2, T, seed=T, min_len=T // 2)
        loss, logp, ol = tr.step(batch, training=False)
        assert torch.isfinite(loss)
    assert len(model.engine.plans) == 3
    assert (2, 64, False, False) in model.engine.plans    # re-built after eviction, most recent


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_two_rank_nccl_step_equals_single_process_step(precision, tmp_path):
    """Utterance-sharded DP (one process per GPU, bucketed NCCL all-reduce overlapped with the backward graphs) == the
    single-process step on the concatenated batch (reference: nn.DataParallel, trainer.py:91-92)."""
    out = tmp_path / 'dp'
    out.mkdir()
    port = 29600 + os.getpid() % 1000
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(port), os.path.join(ROOT, 'tests', 'dp_worker.py'), str(out), precision]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = json.load(open(out / 'result.json'))
    assert res['ranks_equal'], 'replicas diverged'
    assert res['loss0_rel'] < 1e-6, res                 # same forward arithmetic per utterance
    # the exchanged gradient (mean over ranks + regulariser) equals the single-process gradient of the whole batch up to
    # fp32 summation order.  The Adam update's first steps are -lr * sign(g) wherever |g| >> eps = 1e-7, so the ~1e-6 summation
    # noise flips whole +-lr steps on the elements whose true gradient is 0 (biases in front of a LayerNorm): the update is
    # compared on the elements with a significant reference gradient, the parameters themselves with a bound of a few flips
    assert res['grad_rel'] < 1e-5, res
    # Measured (2 x B200, r2): the exchanged step-1 gradient agrees to 1.4e-7 (fp32) / 1.6e-7 (16-bit) of its norm, the
    # two-step update of the significant elements to 0.7 % (fp32) / 8 % (16-bit): the +-lr flips of step 1 on zero-gradient
    # elements change the 16-bit operand packs, which perturbs the bf16 backward pass of step 2 and flips the sign of ~0.7 % of
    # its small gradients -- the update bound of the 16-bit mode is therefore loose, the gradient itself is the check.
    print({k: v for k, v in res.items() if k not in ('losses', 'ref_losses')})
    assert res['sig_frac'] > 0.5 and res['update_rel_sig'] < (5e-2 if precision == 'fp32' else 0.2), res
    assert res['params_rel'] < 2e-3, res
    assert res['loss2_rel'] < (1e-4 if precision == 'fp32' else 2e-2), res
    assert res['used_graph'] and res['buckets'] == 5
