"""Zero-cost architecture proxies: scores of an UNTRAINED candidate from one minibatch (pruning-at-init measures, as the
NAS-Bench-ASR users' proxy code computes them through ``get_prunable_copy``).

    compute_proxies(model, batch) -> {'grad_norm': ..., 'snip': ..., 'synflow': ..., 'jacob_cov': ..., 'nwot': ...}

* grad_norm = sum over scored tensors of ||g||_2 and snip = sum |theta * g|, from ONE forward + backward of the CTC loss
  (get_loss() on the log-softmax logits, output_len = audio_len // 4, no regulariser, dropout off);
* jacob_cov: backward of dlogits = 1, the input gradient J (B, 80*T), score -sum(log(l + 1e-5) + 1 / (l + 1e-5)) over the
  eigenvalues l of corrcoef(J); NaN when a row of J has zero variance;
* synflow: on the norm-free copy (get_prunable_copy(bn=False)) in the fp32 engine mode, every parameter replaced by its
  absolute value, an all-ones (1, 80, T) input, dlogits = 1; score sum |theta * g|;
* nwot (NASWOT, Mellor et al. 2021): from the forward pass alone (dropout off), the binary code of every ReLU20 unit --
  the block convs' and every non-`zero` node op's, m = (0 < z <= 20), the indicator of the unit's LINEAR region, a
  deliberate choice over the classic z > 0, which counts saturated units as active -- gives the kernel matrix
  K[i, j] = number of units, over the frames valid for both utterances, on which utterances i and j have the same code;
  score log|det K| (fp64 slogdet on the host; -inf when K is singular, e.g. for a batch with a duplicated utterance).
  Valid frames of block k: min(T_k, ceil(audio_len / 2^s_k)), s = (0, 0, 1, 2).  K comes from the gate-bit masks a
  grad plan's forward pass already writes (nbasr_gate_gram, exact integer counts); with grad_norm / snip it reuses
  their forward pass;
* zico (ZiCo, Li et al. 2023; opt-in by name, not in MEASURES): the batch is cut into N interleaved splits (utterance b
  goes to split b mod N, each keeps the padded T); g_k is the gradient of split k's CTC loss (as grad_norm's, dropout
  off).  Per parameter, in fp64, m = mean_k g_k, var = mean_k (g_k - m)^2 and, where var > 0 (the N samples are not all
  equal), r = mean_k |g_k| / sqrt(var); R_l = sum r over tensor l and the score is the sum of ln R_l over the tensors
  with R_l > 0 (nbasr_grad_snr over the N snapshots of the flat gradient buffer).  The ratio is large exactly where the
  split gradients nearly agree, so it amplifies the fp32-atomic rounding of the weight-gradient kernels: two runs agree
  less closely than the other measures do (DESIGN.md 7b).

Scored tensors are the ``.weight`` of every Conv1d and Linear (time-reduction and grouped convs, linear edges, classifier);
LSTM, LayerNorm and biases are not scored ("conv and linear layers", as in the pruning-at-init library).  Per-tensor sums
run on the GPU in fp64 (nbasr_param_stats): gradients at initialisation can be ~1e-20, whose squares underflow fp32.
The model's parameters, gradients, Adam state and dropout counter are unchanged on return.
"""
import math

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .model import ASRModel, FEATURES, TR_STRIDES
from .trainer import ctc_loss_cuda

MEASURES = ('grad_norm', 'snip', 'synflow', 'jacob_cov', 'nwot')     # the default set
ACCEPTED = MEASURES + ('zico',)                                        # every measure compute_proxies computes by name
SEG_CHUNK = 16384          # chunk of nbasr_param_stats / nbasr_grad_snr (optim.cu)
ZICO_MAX_SPLITS = 16       # N <= 16 gradient samples per parameter (nbasr_grad_snr)
# s_k of block k: its frames are the input's halved s_k times, (0, 0, 1, 2)
LEN_SHIFT = tuple(sum(1 for s in TR_STRIDES[:k + 1] if s == 2) for k in range(len(TR_STRIDES)))


def parse_measures(text):
    """'grad_norm,snip' -> ('grad_norm', 'snip'); unknown names raise ValueError."""
    names = tuple(n.strip() for n in text.split(',') if n.strip())
    bad = [n for n in names if n not in ACCEPTED]
    if bad or not names:
        raise ValueError(f'unknown proxy measure(s) {bad or text!r}; choose from {",".join(ACCEPTED)}')
    return names


def scored_names(model):
    """Parameter names of the scored tensors, in parameter (module construction) order."""
    return [f'{n}.weight' for n, m in model.named_modules() if isinstance(m, (nn.Conv1d, nn.Linear))]


def _segments(eng, names):
    """Segment table of the named tensors in the engine's flat buffers for nbasr_param_stats / nbasr_grad_snr:
    (offsets, lengths, chunk count, partials, out (nseg, 2) fp64), all on the device."""
    segs = [eng.slices[n] for n in names]
    dev = eng.device
    off = torch.tensor([o for o, _ in segs], dtype=torch.int64, device=dev)
    ln = torch.tensor([n for _, n in segs], dtype=torch.int64, device=dev)
    chunks = sum((n + SEG_CHUNK - 1) // SEG_CHUNK for _, n in segs)
    part = torch.empty(2 * chunks, dtype=torch.float64, device=dev)
    out = torch.empty(len(segs), 2, dtype=torch.float64, device=dev)
    return off, ln, chunks, part, out


def _param_stats(eng, names):
    """{name: (sum g^2, sum |theta g|)} over the engine's flat buffers, fp64."""
    off, ln, chunks, part, out = _segments(eng, names)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(eng.lib.nbasr_param_stats(eng.flat_p.data_ptr(), eng.flat_g.data_ptr(), off.data_ptr(), ln.data_ptr(), len(names),
                                         chunks, part.data_ptr(), out.data_ptr(), st), 'param_stats')
    vals = out.cpu().tolist()
    return {n: tuple(v) for n, v in zip(names, vals)}


def zico_split(batch, splits):
    """The N = `splits` interleaved splits of batch ((audio, audio_len), (targets, targets_len)): utterance b goes to split
    b mod N (the sweep's batches are length-sorted: contiguous slices would differ systematically in length); every split
    keeps the batch's padded T.  2 <= N <= min(B, 16), else ValueError."""
    (audio, audio_len), (targets, targets_len) = batch
    B = audio.shape[0]
    if not 2 <= splits <= min(B, ZICO_MAX_SPLITS):
        raise ValueError(f'zico needs 2 <= splits <= min(B, {ZICO_MAX_SPLITS}) = {min(B, ZICO_MAX_SPLITS)}, got {splits}')
    return [((audio[k::splits], audio_len[k::splits]), (targets[k::splits], targets_len[k::splits])) for k in range(splits)]


def zico_snapshots(model, batch, splits=2):
    """(N, len(flat_g)) fp32 device tensor: row k is the engine's flat gradient of the CTC loss of split k of `batch`
    (zico_split; one forward + backward of a grad plan per split, dropout off).  The model's flat_g is unchanged."""
    parts = zico_split(batch, splits)
    eng = model.engine
    eng.bind()
    dev = eng.device
    with torch.cuda.device(dev):
        snaps = torch.empty(splits, eng.flat_g.numel(), dtype=torch.float32, device=dev)
        saved_g = eng.flat_g.clone()
        try:
            for k, ((audio, audio_len), (targets, targets_len)) in enumerate(parts):
                pl = eng.forward(audio.to(dev, torch.float32).contiguous(), training=False, grad=True)
                ctc_loss_cuda(pl.logp, audio_len.to(dev, torch.int64).contiguous(), 4,
                              targets.to(dev, torch.int32).contiguous(), targets_len.to(dev, torch.int64).contiguous(),
                              dlogits=pl.dlogits)
                eng.backward(pl)
                snaps[k].copy_(eng.flat_g)
        finally:
            eng.flat_g.copy_(saved_g)
    return snaps


def zico_stats(model, snaps):
    """{scored name: (R, n)} from gradient snapshots (N, len(flat_g)): R = sum of mean|g| / std(g) over the n parameters
    whose N samples are not all equal (nbasr_grad_snr, fp64, deterministic)."""
    eng = model.engine
    names = scored_names(model)
    if snaps.dtype != torch.float32 or snaps.dim() != 2 or snaps.stride(1) != 1 or snaps.shape[1] < eng.flat_g.numel():
        raise ValueError('snapshots: a (N, len(flat_g)) fp32 tensor with unit column stride')
    with torch.cuda.device(eng.device):
        off, ln, chunks, part, out = _segments(eng, names)
        _lib.check(eng.lib.nbasr_grad_snr(snaps.data_ptr(), snaps.stride(0), snaps.shape[0], off.data_ptr(), ln.data_ptr(),
                                          len(names), chunks, part.data_ptr(), out.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream), 'grad_snr')
        vals = out.cpu().tolist()
    return {n: tuple(v) for n, v in zip(names, vals)}


def zico_layers(stats):
    """{name: ln R} over the tensors with R > 0 (a tensor with no included parameter contributes nothing)."""
    return {n: math.log(r) for n, (r, _) in stats.items() if r > 0}


def corrcoef_from_gram(G, s, D):
    """corrcoef of the rows of a (B, D) matrix from its Gram matrix G = X X^T and row sums s (float64 numpy)."""
    G, s = np.asarray(G, np.float64), np.asarray(s, np.float64)
    cov = G - np.outer(s, s) / D
    d = np.sqrt(np.diag(cov))
    with np.errstate(divide='ignore', invalid='ignore'):
        c = cov / d[:, None] / d[None, :]
    return np.clip(c, -1.0, 1.0)


def jacob_cov_score(corr):
    """-sum(log(l + k) + 1/(l + k)), k = 1e-5, over the eigenvalues of the correlation matrix; NaN if it has NaNs."""
    corr = np.asarray(corr, np.float64)
    if not np.all(np.isfinite(corr)):
        return float('nan')
    v = np.linalg.eigvalsh(corr)
    k = 1e-5
    return float(-np.sum(np.log(v + k) + 1.0 / (v + k)))


def _row_gram(eng, x, B, D, ld):
    dev = eng.device
    gram = torch.empty(B, B, dtype=torch.float64, device=dev)
    rs = torch.empty(B, dtype=torch.float64, device=dev)
    work = torch.empty(((D + 255) // 256) * (B * (B + 1) // 2 + B), dtype=torch.float64, device=dev)
    _lib.check(eng.lib.nbasr_row_gram(x.data_ptr(), B, D, ld, gram.data_ptr(), rs.data_ptr(), work.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), 'row_gram')
    return gram.cpu().numpy(), rs.cpu().numpy()


def jacob_correlation(model, audio):
    """Correlation matrix (B, B) of the rows of the input gradient of sum(logits) (the jacob_cov statistic)."""
    eng = model.engine
    with torch.cuda.device(eng.device or audio.device):
        pl = eng.forward(audio, training=False, grad=True, input_grad=True)
        pl.dlogits.fill_(1.0)
        eng.backward(pl)
        B, T = pl.B, pl.T
        Tp = pl.in_geo.Tp
        # padded channels-last input gradient: utterance b is Tp * 80 consecutive floats from row b * Tp, its pad rows zero
        G, s = _row_gram(eng, pl.dx_in, B, Tp * FEATURES, Tp * FEATURES)
    return corrcoef_from_gram(G, s, FEATURES * T)


def gate_frames(audio_len, T_k, s_k):
    """Valid frames of a block with T_k frames and length shift s_k: min(T_k, ceil(audio_len / 2^s_k))."""
    return min(T_k, -(-int(audio_len) >> s_k))


def _gate_table(eng, pl):
    """The plan's ReLU layers as a device array of nbasr_gate_layer, built on first use and kept on the plan."""
    if getattr(pl, 'gate_table', None) is None:
        arr = (_lib.GateLayer * len(pl.gates))()
        for e, (mask, geo, k) in zip(arr, pl.gates):
            e.mask, e.mask_rows, e.w, e.C = mask.t.data_ptr(), geo.rows, mask.w, geo.C
            e.Tp, e.T, e.s = geo.Tp, geo.T, LEN_SHIFT[k]
        pl.gate_table = torch.frombuffer(bytearray(arr), dtype=torch.uint8).to(eng.device)
    return pl.gate_table


def _gate_gram(eng, pl, audio_len):
    """K (B, B) uint64 numpy from the gate masks of a grad plan's last forward pass; audio_len int64 on the device."""
    table = _gate_table(eng, pl)
    B = pl.B
    K = torch.empty(B, B, dtype=torch.int64, device=eng.device)
    work = torch.empty(int(eng.lib.nbasr_gate_gram_work_elems(B)), dtype=torch.int64, device=eng.device)
    _lib.check(eng.lib.nbasr_gate_gram(table.data_ptr(), len(pl.gates), audio_len.data_ptr(), B, K.data_ptr(), work.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream), 'gate_gram')
    return K.cpu().numpy().view(np.uint64)


def nwot_kernel(model, batch):
    """NASWOT kernel matrix K (B, B) uint64 of `model` on batch ((audio, audio_len), ...): one forward pass of a grad
    plan, dropout off, no backward."""
    eng = model.engine
    eng.bind()
    (audio, audio_len) = batch[0]
    with torch.cuda.device(eng.device):
        alen = audio_len.to(eng.device, torch.int64).contiguous()
        pl = eng.forward(audio.to(eng.device, torch.float32).contiguous(), training=False, grad=True)
        return _gate_gram(eng, pl, alen)


def nwot_score(K):
    """log|det K| in fp64 (numpy.linalg.slogdet); -inf when K is singular."""
    return float(np.linalg.slogdet(np.asarray(K, dtype=np.float64))[1])


def _norm_free_fp32_copy(model):
    """The parameters of model.get_prunable_copy(bn=False) on the fp32 engine.  The module tree is built on the meta device
    and takes the model's tensors (the engine copies them into its own flat buffer when it binds): no host-side default
    initialisation, which costs 0.3-0.6 s per candidate."""
    with torch.device('meta'):
        new = ASRModel(model.arch_desc, num_classes=model.num_classes, use_rnn=model.use_rnn, use_norm=False,
                       dropout_rate=model.dropout_rate, precision='fp32')
    new.load_state_dict(model.state_dict(), strict=False, assign=True)
    new.engine.bind()
    return new


def synflow_stats(model, T, copy=None):
    """{scored name: sum |theta g|} of synflow.  `copy`: a norm-free fp32 model to run on (default: built from `model`)."""
    net = copy if copy is not None else _norm_free_fp32_copy(model)
    eng = net.engine
    eng.bind()
    names = scored_names(net)
    with torch.cuda.device(eng.device):
        saved_p, saved_g = eng.flat_p.clone(), eng.flat_g.clone()
        try:
            eng.flat_p.abs_()
            eng.refresh_packs(force=True)
            ones = torch.ones(1, FEATURES, T, dtype=torch.float32, device=eng.device)
            pl = eng.forward(ones, training=False, grad=True)
            pl.dlogits.fill_(1.0)
            eng.backward(pl)
            st = _param_stats(eng, names)
        finally:
            # restore the exact bits (not sign * |theta|: -0.0 and the 64-element pads stay as they were) and the packs
            eng.flat_p.copy_(saved_p)
            eng.flat_g.copy_(saved_g)
            eng.refresh_packs(force=True)
    if copy is None:
        net._engine = None           # engine <-> model is a reference cycle: free the copy's device memory now
    return {n: v[1] for n, v in st.items()}


def compute_proxies(model, batch, measures=MEASURES, per_layer=False, zico_splits=2):
    """Zero-cost proxies of `model` on one batch ((audio (B,80,T), audio_len), (targets, targets_len)).  `measures`: names
    from ACCEPTED (default MEASURES; zico only when named, over `zico_splits` interleaved splits).

    Returns {measure: float}, or with per_layer=True {measure: {parameter name: float}} for grad_norm / snip / synflow /
    zico (zico: ln R of the contributing tensors only; jacob_cov and nwot are whole-network scores and stay floats)."""
    measures = tuple(measures)
    bad = [m for m in measures if m not in ACCEPTED]
    if bad:
        raise ValueError(f'unknown proxy measure(s) {bad}; choose from {ACCEPTED}')
    if 'zico' in measures:
        zico_split(batch, zico_splits)               # an invalid split count fails before any GPU work
    eng = model.engine
    eng.bind()
    dev = eng.device
    (audio, audio_len), (targets, targets_len) = batch
    out = {}
    with torch.cuda.device(dev):
        audio = audio.to(dev, torch.float32).contiguous()
        saved_g = eng.flat_g.clone()
        pl = None
        try:
            if 'grad_norm' in measures or 'snip' in measures:
                pl = eng.forward(audio, training=False, grad=True)
                ctc_loss_cuda(pl.logp, audio_len.to(dev, torch.int64).contiguous(), 4,
                              targets.to(dev, torch.int32).contiguous(), targets_len.to(dev, torch.int64).contiguous(),
                              dlogits=pl.dlogits)
                eng.backward(pl)
                st = _param_stats(eng, scored_names(model))
                if 'grad_norm' in measures:
                    out['grad_norm'] = {n: math.sqrt(v[0]) for n, v in st.items()}
                if 'snip' in measures:
                    out['snip'] = {n: v[1] for n, v in st.items()}
            if 'jacob_cov' in measures:
                out['jacob_cov'] = jacob_cov_score(jacob_correlation(model, audio))
            if 'nwot' in measures:
                # the backward pass only reads the gate masks: grad_norm / snip's forward pass is reused as it stands
                alen = audio_len.to(dev, torch.int64).contiguous()
                if pl is None:
                    pl = eng.forward(audio, training=False, grad=True)
                out['nwot'] = nwot_score(_gate_gram(eng, pl, alen))
        finally:
            eng.flat_g.copy_(saved_g)
        if 'synflow' in measures:
            out['synflow'] = synflow_stats(model, audio.shape[2])
        if 'zico' in measures:
            # after the other measures: their plans and passes run exactly as without zico
            out['zico'] = zico_layers(zico_stats(model, zico_snapshots(model, batch, zico_splits)))
    res = {}
    for m in measures:
        v = out[m]
        res[m] = v if (per_layer or not isinstance(v, dict)) else float(sum(v.values()))
    return res
