"""fp64 CPU restatement of the zero-cost proxies (grad_norm, snip, synflow, jacob_cov) with torch autograd on
oracle/model_ref.forward.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Same definitions as nb_asr_b200/proxies.py, following the pruning-at-init
library's measures: scored tensors are the `.weight` of every Conv1d and Linear (module_order kinds 'conv' / 'linear');
LSTM, LayerNorm and biases are not scored.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import model_ref as M


def scored_keys(arch, use_rnn=True):
    return [f'{prefix}.weight' for prefix, kind, _ in M.module_order(arch, use_rnn) if kind in ('conv', 'linear')]


def _p64(sd, fn=None):
    return {k: (fn(v) if fn else v).detach().double().clone().requires_grad_(True) for k, v in sd.items()}


def grad_stats(sd, arch, audio, audio_len, targets, targets_len, use_rnn=True):
    """{key: (||g||_2, sum |theta g|)} of the CTC loss (log-softmax logits, output_len = audio_len // 4)."""
    p = _p64(sd)
    logits = M.forward(p, arch, audio.double(), use_rnn)
    loss = M.ctc_loss_ref(F.log_softmax(logits, dim=2), audio_len // 4, targets, targets_len)
    loss.backward()
    out = {}
    for k in scored_keys(arch, use_rnn):
        g = p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])
        out[k] = (float(g.norm()), float((p[k].detach() * g).abs().sum()))
    return out


def jacob_corr(sd, arch, audio, use_rnn=True):
    """corrcoef of the rows of d sum(logits) / d audio, (B, 80*T)."""
    p = {k: v.detach().double() for k, v in sd.items()}
    x = audio.double().clone().requires_grad_(True)
    y = M.forward(p, arch, x, use_rnn)
    y.backward(torch.ones_like(y))
    J = x.grad.reshape(x.shape[0], -1).numpy()
    return np.corrcoef(J), x.grad


def jacob_cov_score(corr):
    v, _ = np.linalg.eig(corr)
    k = 1e-5
    return float(-np.sum(np.log(v + k) + 1.0 / (v + k)).real)


def synflow(sd, arch, T, use_rnn=True):
    """{key: sum |theta g|} on the norm-free network (use_norm=False), |theta| for every parameter, ones (1, 80, T) input."""
    p = _p64({k: v for k, v in sd.items() if '.norm_layer.' not in k}, torch.abs)
    y = M.forward(p, arch, torch.ones(1, M.FEATURES, T, dtype=torch.float64), use_rnn, use_norm=False)
    y.sum().backward()
    out = {}
    for k in scored_keys(arch, use_rnn):
        g = p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])
        out[k] = float((p[k].detach() * g).abs().sum())
    return out
