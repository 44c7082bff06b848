"""fp64 CPU restatement of the ZiCo proxy (`zico`, Li et al. 2023) with torch autograd on oracle/model_ref.forward.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Same definition as nb_asr_b200/proxies.py: utterance b of the batch goes
to split b mod N (each split keeps the padded T), g_k is the gradient of split k's CTC loss (log-softmax logits,
output_len = audio_len // 4, batch mean), scored tensors as in proxies_ref.scored_keys.

* snr_stats: the per-tensor (R, count) of the definition (fp64, two-pass population variance, included iff var > 0),
  the statistic nbasr_grad_snr computes;
* caculate_zico: a direct transcription of the official `caculate_zico` (np.std, np.nonzero, tmpsum == 0 skipped,
  np.log), on {name: (N, P) array}.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import model_ref as M
from .proxies_ref import _p64, scored_keys


def split_grads(sd, arch, audio, audio_len, targets, targets_len, splits=2, use_rnn=True):
    """{key: (N, P) fp64 numpy}: row k is the flattened gradient of the CTC loss of split k (utterances k, k + N, ...)."""
    rows = {k: [] for k in scored_keys(arch, use_rnn)}
    for s in range(splits):
        p = _p64(sd)
        logits = M.forward(p, arch, audio[s::splits].double(), use_rnn)
        loss = M.ctc_loss_ref(F.log_softmax(logits, dim=2), audio_len[s::splits] // 4, targets[s::splits],
                              targets_len[s::splits])
        loss.backward()
        for k in rows:
            g = p[k].grad if p[k].grad is not None else torch.zeros_like(p[k])
            rows[k].append(g.detach().reshape(-1).numpy())
    return {k: np.stack(v) for k, v in rows.items()}


def snr_stats(G):
    """(R, count) of one tensor's samples G (N, P): per parameter m = sum g / N, var = sum (g - m)^2 / N in fp64; over the
    parameters with var > 0, R = sum (sum |g| / N) / sqrt(var) and count = their number."""
    G = np.asarray(G, np.float64)
    N = G.shape[0]
    m = G.sum(0) / N
    var = ((G - m) ** 2).sum(0) / N
    inc = var > 0
    r = (np.abs(G).sum(0)[inc] / N) / np.sqrt(var[inc])
    return float(r.sum()), int(inc.sum())


def zico_layers(grads):
    """{key: ln R} over the tensors with R > 0, from {key: (N, P) samples}."""
    out = {}
    for k, G in grads.items():
        R, _ = snr_stats(G)
        if R > 0:
            out[k] = float(np.log(R))
    return out


def caculate_zico(grad_dict):
    """The official ZiCo score (ZiCo repository, `caculate_zico`), transcribed: {name: (N, P) gradient samples}."""
    for i, modname in enumerate(grad_dict.keys()):
        grad_dict[modname] = np.array(grad_dict[modname])
    nsr_mean_sum_abs = 0
    for j, modname in enumerate(grad_dict.keys()):
        nsr_std = np.std(grad_dict[modname], axis=0)
        nonzero_idx = np.nonzero(nsr_std)[0]
        nsr_mean_abs = np.mean(np.abs(grad_dict[modname]), axis=0)
        tmpsum = np.sum(nsr_mean_abs[nonzero_idx] / nsr_std[nonzero_idx])
        if tmpsum == 0:
            pass
        else:
            nsr_mean_sum_abs += np.log(tmpsum)
    return nsr_mean_sum_abs
