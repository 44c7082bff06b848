"""Train / eval step on the B200 engine behind the reference Trainer API.

Mirrors nasbench_asr/training/torch/trainer.py: get_loss (:36-44), Trainer.step (:208-227),
Trainer.decode (:229-247, with the greedy decoder of tf/metrics/ctc.py:76-81 in place of the
third-party beam search, as BASELINE.json's north_star asks), train (:80-206), save/load
(:249-258), remember_best/recall_best (:260-264), AvgMeter (:16-33).

Differences that are deliberate: the step is one fused pipeline (forward plan -> CTC kernel ->
backward plan -> [NCCL all-reduce] -> regulariser+clip+Adam kernel) with no autograd graph and
no host synchronisation; data-parallel training is one process per GPU (torch.distributed)
instead of single-process nn.DataParallel (:91-92).
"""
import collections
import collections.abc as cabc
import pathlib

import numpy as np
import os

import torch

from . import _lib
from .model import PadConvRelu, print_model_summary


class AvgMeter:
    def __init__(self):
        self.reset()

    def reset(self):
        self.avg = 0
        self.n = 0

    def update(self, a):
        if not self.n:
            self.avg, self.n = a, 1
        else:
            self.avg = self.avg * (self.n / (self.n + 1)) + (a / (self.n + 1))
            self.n += 1

    def get(self):
        return self.avg


class _Ws:
    pass


class _CtcWorkspace:
    """Per-shape scratch buffers for loss() / decode() called on free-standing tensors (bounded LRU).  The step itself
    keeps its workspaces on the engine plan (`plan.ws`), so pointers captured in CUDA graphs live exactly as long as
    the plan and the graphs do."""
    MAX = 16

    def __init__(self):
        self.cache = collections.OrderedDict()

    @staticmethod
    def make(dev, B, T, V, S, arena=None):
        """arena: the engine plan's arena (zero-filled device memory): one carve instead of nine allocations + fills"""
        L = 2 * S + 1
        z = arena.zeros if arena is not None else (lambda shape, dtype: torch.zeros(shape, dtype=dtype, device=dev))
        w = _Ws()
        w.work = z(2 * B * T * L + 16, torch.float32)
        w.nll = z(B, torch.float32)
        w.loss = z(1, torch.float32)
        w.dlogits = z((B, T, V), torch.float32)
        w.hyp = z((B, T), torch.int32)
        w.hyp_len = z(B, torch.int32)
        w.dist = z(B, torch.int32)
        w.per = z(2, torch.float64)
        w.iwork = z(B * (S + 2) + 16, torch.int32)
        return w

    def get(self, dev, B, T, V, S):
        key = (str(dev), B, T, V, S)
        w = self.cache.get(key)
        if w is None:
            while len(self.cache) >= self.MAX:
                self.cache.popitem(last=False)
            w = self.cache[key] = self.make(dev, B, T, V, S)
        else:
            self.cache.move_to_end(key)
        return w


_ws = _CtcWorkspace()


def ctc_loss_cuda(logp, output_len_src, len_div, targets, targets_len, dlogits=None):
    """CTC NLL / output_len, batch mean (zero_infinity) on libnbasr; optional d/dlogits."""
    lib = _lib.load()
    B, T, V = logp.shape
    S = targets.shape[1]
    with torch.cuda.device(logp.device):
        ws = _ws.get(logp.device, B, T, V, S)
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.nbasr_ctc(logp.data_ptr(), B, T, V, targets.data_ptr(), S, output_len_src.data_ptr(), len_div,
                                 targets_len.data_ptr(), ws.nll.data_ptr(), ws.loss.data_ptr(),
                                 dlogits.data_ptr() if dlogits is not None else None, ws.work.data_ptr(), st), 'ctc')
    return ws.loss, ws.nll


Alignment = collections.namedtuple('Alignment', 'labels tok start end score')
Alignment.__doc__ = """CTC forced alignment of a batch (nbasr_ctc_align, include/nbasr.h), device tensors:
labels (B,T) int32 class of each output frame on the best path (0 = blank), tok (B,T) int32 index of the target token
the frame emits (-1 on blanks), start / end (B,S) int32 half-open frame span of each target token, score (B,) fp32
best path log-probability (-inf: the row has no path; NaN: a target id outside [1, V)).  -1 marks frames past the
output length, tokens past the target length and every output of a row without a path."""


def ctc_align_cuda(logp, output_len_src, len_div, targets, targets_len):
    """Viterbi alignment of targets (B,S) int32 through logp (B,T,V) fp32 on libnbasr, with output frames
    min(T, output_len_src // len_div) and min(S, targets_len) tokens per row (int64 lengths; all inputs contiguous on one
    device) -> Alignment.  No host synchronisation."""
    lib = _lib.load()
    B, T, V = logp.shape
    S = targets.shape[1]
    dev = logp.device
    with torch.cuda.device(dev):
        i32 = dict(dtype=torch.int32, device=dev)
        out = Alignment(torch.empty((B, T), **i32), torch.empty((B, T), **i32), torch.empty((B, S), **i32),
                        torch.empty((B, S), **i32), torch.empty(B, dtype=torch.float32, device=dev))
        nwork = lib.nbasr_ctc_align_work_bytes(B, T, S)
        work = torch.empty(nwork, dtype=torch.uint8, device=dev) if nwork > 0 else None
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.nbasr_ctc_align(logp.data_ptr(), B, T, V, targets.data_ptr(), S, output_len_src.data_ptr(), len_div,
                                       targets_len.data_ptr(), *(t.data_ptr() for t in out),
                                       work.data_ptr() if work is not None else None, st), 'ctc_align')
    return out


EditAlignment = collections.namedtuple('EditAlignment', 'counts ref_at hyp_at confusion')
EditAlignment.__doc__ = """Phone error breakdown of a decoded batch (nbasr_edit_align, include/nbasr.h), device tensors:
counts (B,4) int32 [hits, substitutions, deletions, insertions], ref_at (B,H) int32 reference position aligned to each
hypothesis position (-1: insertion), hyp_at (B,S) int32 hypothesis position aligned to each reference position (-1:
deletion), confusion (V,V) int64 view of the uint64 counts confusion[ref class, hyp class] (row 0: insertions, column 0:
deletions).  A row with an id out of range has counts and alignments -1 and adds nothing to confusion."""

ErrorReport = collections.namedtuple('ErrorReport', 'per counts ref_at hyp_at confusion')
ErrorReport.__doc__ = """Trainer.error_report: per (the value Trainer.decode returns) and the EditAlignment fields."""


def edit_align_cuda(hyp, hyp_len, targets, targets_len, lut, V, confusion=None):
    """Levenshtein alignment of the folded hypotheses hyp (B,H) int32 / hyp_len (B,) int32, as nbasr_greedy_per writes
    them, against targets (B,S) int32 / targets_len (B,) int64 mapped through lut (V,) int32 or None, on libnbasr (all
    inputs contiguous on one device) -> EditAlignment.  confusion: an int64 (V,V) accumulator the counts are added to;
    None starts from zeros.  No host synchronisation."""
    lib = _lib.load()
    B, H = hyp.shape
    S = targets.shape[1]
    dev = hyp.device
    with torch.cuda.device(dev):
        if confusion is None:
            confusion = torch.zeros((V, V), dtype=torch.int64, device=dev)
        elif confusion.shape != (V, V) or confusion.dtype != torch.int64 or confusion.device != dev or not confusion.is_contiguous():
            raise ValueError(f'edit_align: confusion must be a contiguous int64 ({V}, {V}) tensor on {dev}')
        i32 = dict(dtype=torch.int32, device=dev)
        counts, ref_at, hyp_at = torch.empty((B, 4), **i32), torch.empty((B, H), **i32), torch.empty((B, S), **i32)
        nwork = lib.nbasr_edit_align_work_bytes(B, H, S)
        work = torch.empty(nwork, dtype=torch.uint8, device=dev) if nwork > 0 else None
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(lib.nbasr_edit_align(hyp.data_ptr(), hyp_len.data_ptr(), H, targets.data_ptr(), S, targets_len.data_ptr(),
                                        lut.data_ptr() if lut is not None else None, B, V, counts.data_ptr(),
                                        ref_at.data_ptr(), hyp_at.data_ptr(), confusion.data_ptr(),
                                        work.data_ptr() if work is not None else None, st), 'edit_align')
    return EditAlignment(counts, ref_at, hyp_at, confusion)


class _CtcLossFn(torch.autograd.Function):
    """Differentiable wrapper for users who call loss() on a tensor that requires grad."""

    @staticmethod
    def forward(ctx, output, output_len, targets, targets_len):
        out = output.detach().contiguous().float()
        olen = output_len.to(out.device, torch.int64).contiguous()
        d = torch.empty_like(out)
        loss, nll = ctc_loss_cuda(out, olen, 1, targets.to(out.device, torch.int32).contiguous(),
                                  targets_len.to(out.device, torch.int64).contiguous(), dlogits=d)
        # the kernel emits d/dlogits = (softmax - occupancy) * s with s = 1/(B*len); the gradient wrt the
        # log-probs themselves is -occupancy * s = d - softmax * s on active rows, 0 elsewhere.
        B, T, _ = out.shape
        s = 1.0 / (olen.clamp(min=1).float() * B)
        active = (torch.arange(T, device=out.device)[None, :] < olen[:, None]) & (nll > 0)[:, None]
        ctx.save_for_backward((d - out.exp() * s[:, None, None]) * active[:, :, None])
        return loss.clone().squeeze(0)

    @staticmethod
    def backward(ctx, g):
        (dlogp,) = ctx.saved_tensors
        return dlogp * g, None, None, None


def get_loss():
    """loss(output (B,T',49) log-probs, output_len, targets, targets_len) -> scalar (trainer.py:36-44)."""
    def loss(output, output_len, targets, targets_len):
        if not output.is_cuda:
            raise RuntimeError('nb_asr_b200 loss runs on a CUDA device only (no CPU fallback)')
        if output.requires_grad and torch.is_grad_enabled():
            return _CtcLossFn.apply(output, output_len, targets, targets_len)
        out = output.detach().contiguous().float()
        l, _ = ctc_loss_cuda(out, output_len.to(out.device, torch.int64).contiguous(), 1,
                             targets.to(out.device, torch.int32).contiguous(),
                             targets_len.to(out.device, torch.int64).contiguous())
        return l.clone().squeeze(0)
    return loss


class _GraphCaptureError(RuntimeError):
    pass


class FusedAdam:
    """Handle on the engine-resident Adam state with a torch.optim.Adam-shaped state_dict."""

    def __init__(self, model, lr, eps=1e-7, betas=(0.9, 0.999)):
        self.model, self.eps, self.betas = model, eps, betas
        self.param_groups = [dict(lr=lr, betas=betas, eps=eps, weight_decay=0, amsgrad=False)]

    @property
    def lr(self):
        return self.param_groups[0]['lr']

    def zero_grad(self, set_to_none=False):
        self.model.engine.bind()
        self.model.engine.flat_g.zero_()

    def _views(self, flat):
        eng = self.model.engine
        out = []
        for name, p in zip(eng.names, eng.params):
            off, n = eng.slices[name]
            v = flat[off:off + n]
            if eng._is_dense_conv_w(name):
                co, ci, k = p.shape
                out.append(v.view(co, k, ci).permute(0, 2, 1))
            else:
                out.append(v.view(p.shape))
        return out

    def state_dict(self):
        eng = self.model.engine
        eng.bind()
        step = float(eng.opt_state[0].item())
        m, v = self._views(eng.adam_m), self._views(eng.adam_v)
        state = {i: dict(step=torch.tensor(step), exp_avg=m[i].contiguous().clone(), exp_avg_sq=v[i].contiguous().clone())
                 for i in range(len(m))} if step > 0 else {}
        groups = [dict(self.param_groups[0], params=list(range(len(m))))]
        return dict(state=state, param_groups=groups)

    def load_state_dict(self, sd):
        eng = self.model.engine
        eng.bind()
        m, v = self._views(eng.adam_m), self._views(eng.adam_v)
        step = 0.0
        for i, s in sd.get('state', {}).items():
            m[int(i)].copy_(s['exp_avg'])
            v[int(i)].copy_(s['exp_avg_sq'])
            step = float(s['step'])
        eng.opt_state[0:1].fill_(step)
        if sd.get('param_groups'):
            self.param_groups[0]['lr'] = sd['param_groups'][0]['lr']


class ExponentialLR:
    def __init__(self, optimizer, gamma):
        self.optimizer, self.gamma = optimizer, gamma

    def step(self):
        self.optimizer.param_groups[0]['lr'] *= self.gamma


def set_time_limit(loader, time_limit):
    """training/torch/timit.py:116-119 when the loader exposes the same hooks; otherwise a no-op."""
    db = getattr(loader, 'dataset', None)
    sampler = getattr(loader, 'sampler', None)
    if db is not None and sampler is not None and hasattr(db, 'get_indices_shorter_than'):
        sampler.indices = db.get_indices_shorter_than(time_limit)


class Trainer:
    def __init__(self, dataloaders, loss, gpus=None, save_dir=None, verbose=True):
        encoder, train_load, valid_load, test_load = dataloaders
        self.encoder = encoder
        self.train_load, self.valid_load, self.test_load = train_load, valid_load, test_load
        self.gpus = gpus
        self.save_dir = pathlib.Path(save_dir) if save_dir else save_dir
        if self.save_dir:
            self.save_dir.mkdir(exist_ok=True, parents=True)
        self.verbose = verbose
        self.loss = loss
        if self.gpus is not None and (not isinstance(self.gpus, cabc.Sequence) or bool(self.gpus)):
            if not isinstance(gpus, cabc.Sequence):
                self.gpus = [self.gpus]
            self.device = torch.device(f'cuda:{self.gpus[0]}')
        else:
            raise RuntimeError('the b200 backend needs gpus=[device index]: there is no CPU execution path')
        self.fold_to = 39
        lut = encoder.fold_lut(self.fold_to) if encoder is not None and hasattr(encoder, 'fold_lut') else None
        self._lut = torch.as_tensor(lut, dtype=torch.int32, device=self.device) if lut is not None else None
        self.model = None
        self._model = None
        self.lr = None
        self.optimizer = None
        self.scheduler = None
        self._best_weights = None
        self.last_hyp = None

    # ---------------------------------------------------------------- the unit of work
    def step(self, inputs, training):
        """((audio (B,80,T) f32, audio_len (B,)), (targets (B,S) i32, targets_len (B,))) ->
        (loss w/o regulariser, log-probs (B,T',49), output_len), all detached (trainer.py:208-227)."""
        (audio, audio_len), (targets, targets_len) = inputs
        dev = self.device
        with torch.cuda.device(dev):      # libnbasr launches on the CURRENT stream: make gpus[0] the current device
            audio = audio.to(device=dev, dtype=torch.float32, non_blocking=True)
            audio_len = audio_len.to(device=dev, dtype=torch.int64, non_blocking=True)
            targets = targets.to(device=dev, dtype=torch.int32, non_blocking=True).contiguous()
            targets_len = targets_len.to(device=dev, dtype=torch.int64, non_blocking=True)
            if getattr(self, 'use_graph', False):
                try:
                    return self._step_graph(audio, audio_len, targets, targets_len, training)
                except _GraphCaptureError as e:       # eager launches of the same kernels; still GPU-only
                    import sys
                    sys.stderr.write(f'[nb_asr_b200] CUDA graph capture unavailable ({e}); running eagerly\n')
                    self.use_graph = False
            return self._step_eager(audio, audio_len, targets, targets_len, training)

    def _lr(self):
        return self.optimizer.param_groups[0]['lr'] if self.optimizer is not None else (self.lr or 1e-4)

    @staticmethod
    def _plan_ws(pl, dev, B, S):
        """CTC / decode workspace of this (plan, S): owned by the plan, so it lives as long as graphs captured on it."""
        ws = pl.ws.get(S)
        if ws is None:
            ws = pl.ws[S] = _CtcWorkspace.make(dev, B, pl.Tq, pl.V, S, arena=pl.arena)
        return ws

    def _ctc(self, eng, pl, targets, audio_len, targets_len, training, ws):
        B, S = targets.shape
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(eng.lib.nbasr_ctc(pl.logp.data_ptr(), B, pl.Tq, pl.V, targets.data_ptr(), S, audio_len.data_ptr(), 4,
                                     targets_len.data_ptr(), ws.nll.data_ptr(), ws.loss.data_ptr(),
                                     pl.dlogits.data_ptr() if training else None, ws.work.data_ptr(), st), 'ctc')
        eng.launches += 1

    def _step_eager(self, audio, audio_len, targets, targets_len, training):
        model = self._model
        eng = model.engine
        pl = eng.forward(audio, training=model.training, grad=training)
        B, S = targets.shape
        ws = self._plan_ws(pl, self.device, B, S)
        self._ctc(eng, pl, targets, audio_len, targets_len, training, ws)
        if training:
            eng.backward(pl)
            self._allreduce_grads(eng)
            eng.optimizer_step(self._lr())
        return ws.loss[0].clone(), pl.logp.clone(), audio_len // 4

    def _step_graph(self, audio, audio_len, targets, targets_len, training):
        """Same launches as _step_eager, replayed from CUDA graphs (static buffers, no per-launch host cost).  The graphs
        are stored ON the engine plan they were captured on (plan.graphs), so they can never outlive its buffers or be
        replayed against another engine."""
        import torch.distributed as dist
        model = self._model
        eng = model.engine
        eng.bind()
        B, _, T = audio.shape
        S = targets.shape[1]
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        pl = eng.plan(B, T, model.training, training)
        key = (S, bool(training), multi)
        ent = pl.graphs.get(key)
        ws = self._plan_ws(pl, self.device, B, S)
        eng.refresh_packs()
        if training:
            eng.set_lr(self._lr())
        if ent is None:
            ent = dict(alen=torch.zeros_like(audio_len), tg=torch.zeros_like(targets), tl=torch.zeros_like(targets_len), ws=ws)
            ent['alen'].copy_(audio_len); ent['tg'].copy_(targets); ent['tl'].copy_(targets_len)
            pl.audio.copy_(audio)

            def body_main(bwd_upto=None):
                if model.training and eng.training_drop > 0:
                    eng.drop_step.add_(1)
                eng._run(pl.fwd)
                self._ctc(eng, pl, ent['tg'], ent['alen'], ent['tl'], training, ws)
                if training:
                    eng.flat_g.zero_()
                    eng._run(pl.bwd if bwd_upto is None else pl.bwd[:bwd_upto])
                    if not multi:
                        eng._optimizer_launch()

            # eager warm-up run on a side stream (sets function attributes, fills the tensor-map cache); its effect on
            # the parameters, the optimiser state and the dropout counter is rolled back afterwards
            state = eng.snapshot_state() if (training or model.training) else None
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                body_main()
                if training and multi:
                    eng._optimizer_launch()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            if state is not None:
                eng.restore_state(state)
            n0 = eng.launches
            try:
                g1 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g1):
                    body_main()
                ent['g1'] = g1
                ent['n1'] = eng.launches - n0
                if training and multi:
                    n0 = eng.launches
                    g2 = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g2):
                        eng._optimizer_launch()
                    ent['g2'] = g2
                    ent['n2'] = eng.launches - n0
                    if os.environ.get('NBASR_DP_BUCKETS', '1') != '0' and len(pl.buckets) > 1:
                        # bucketed exchange: the backward pass is cut where a contiguous range of the flat gradient becomes
                        # final (head + LSTM, then blocks 3..0); each range is all-reduced on NCCL's stream while the next
                        # segment of the backward pass runs (SURVEY.md 8e: "launched bucket-wise during backward").
                        marks = [m for m, _, _ in pl.buckets]
                        segs = []
                        for k in range(1, len(marks)):
                            gk = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(gk):
                                eng._run(pl.bwd[marks[k - 1]:marks[k]])
                            segs.append(gk)
                        eng.launches = n0 + ent['n2']          # the segments re-capture calls g1 already counted
                        g0 = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g0):
                            body_main(bwd_upto=marks[0])
                        eng.launches = n0 + ent['n2']
                        ent['g0'], ent['segs'] = g0, segs
            except Exception as e:  # noqa: BLE001
                torch.cuda.synchronize()
                raise _GraphCaptureError(str(e)) from e
            pl.graphs[key] = ent
        ent['alen'].copy_(audio_len, non_blocking=True)
        ent['tg'].copy_(targets, non_blocking=True)
        ent['tl'].copy_(targets_len, non_blocking=True)
        pl.audio.copy_(audio, non_blocking=True)
        if training and multi and 'segs' in ent:
            from .distributed import allreduce_mean_async
            works = []
            for k, g in enumerate([ent['g0']] + ent['segs']):
                g.replay()
                _, lo, hi = pl.buckets[k]
                works.append(allreduce_mean_async(eng.flat_g[lo:hi]))
            for w in works:
                w.wait()                                   # stream-side wait: the optimiser graph follows the last bucket
            eng.launches += ent['n1']
            ent['g2'].replay()
            eng.launches += ent['n2']
            return ws.loss[0].clone(), pl.logp.clone(), audio_len // 4
        ent['g1'].replay()
        eng.launches += ent['n1']
        if training and multi:
            self._allreduce_grads(eng)
            ent['g2'].replay()
            eng.launches += ent['n2']
        return ws.loss[0].clone(), pl.logp.clone(), audio_len // 4

    def _allreduce_grads(self, eng):
        from .distributed import allreduce_mean_
        allreduce_mean_(eng.flat_g)

    def decode(self, output, output_len, val_inputs, beam_width=None):
        """CTC decode + 48->39 fold + PER (batch mean of edit_distance / ref_len).

        Default (north_star): greedy decode.  ``beam_width=12`` (or ``trainer.beam_width = 12``) runs the prefix beam
        search the reference's CTCBeamDecoder performs (trainer.py:71,236) -- see nbasr_beam_per."""
        with torch.cuda.device(self.device):
            return self._decode(output, output_len, val_inputs, beam_width)

    def _decode(self, output, output_len, val_inputs, beam_width):
        _, (targets, targets_len) = val_inputs
        dev = self.device
        targets = targets.to(device=dev, dtype=torch.int32).contiguous()
        targets_len = targets_len.to(device=dev, dtype=torch.int64)
        output = output.to(device=dev).contiguous().float()
        output_len = output_len.to(device=dev, dtype=torch.int64)
        B, T, V = output.shape
        S = targets.shape[1]
        ws = _ws.get(dev, B, T, V, S)
        lib = _lib.load()
        st = torch.cuda.current_stream().cuda_stream
        bw = beam_width if beam_width is not None else getattr(self, 'beam_width', None)
        lut = self._lut.data_ptr() if self._lut is not None else None
        if bw:
            raw = torch.empty((B, T), dtype=torch.int32, device=dev)
            raw_len = torch.empty((B,), dtype=torch.int32, device=dev)
            _lib.check(lib.nbasr_beam_per(output.data_ptr(), B, T, V, output_len.data_ptr(), 1, int(bw), 40, targets.data_ptr(), S,
                                          targets_len.data_ptr(), lut, raw.data_ptr(), raw_len.data_ptr(), ws.hyp.data_ptr(),
                                          ws.hyp_len.data_ptr(), ws.dist.data_ptr(), ws.per.data_ptr(), ws.iwork.data_ptr(), st),
                       'beam_per')
            self.last_beam = (raw, raw_len)
        else:
            _lib.check(lib.nbasr_greedy_per(output.data_ptr(), B, T, V, output_len.data_ptr(), 1, targets.data_ptr(), S,
                                            targets_len.data_ptr(), lut, ws.hyp.data_ptr(), ws.hyp_len.data_ptr(),
                                            ws.dist.data_ptr(), ws.per.data_ptr(), ws.iwork.data_ptr(), st), 'greedy_per')
        self.last_hyp = (ws.hyp, ws.hyp_len, ws.dist)
        return ws.per[0].clone()

    def align(self, output, output_len, val_inputs):
        """CTC forced alignment of the batch's targets through the log-probs ``output`` (B,T',49) of ``step``; ``output_len``
        in output frames (one output frame = 4 input frames of 10 ms).  Same arguments as ``decode``:
            loss, logp, out_len = trainer.step(batch, training=False); ali = trainer.align(logp, out_len, batch)
        -> trainer.Alignment of device tensors (see ctc_align_cuda).  Target ids outside [1, V) raise ValueError when the
        targets are host tensors (checked before the upload); on the device such a row comes back with score NaN."""
        _, (targets, targets_len) = val_inputs
        V = output.shape[2]
        if not targets.is_cuda:
            live = torch.arange(targets.shape[1])[None, :] < torch.as_tensor(targets_len).cpu()[:, None]
            if bool((((targets < 1) | (targets >= V)) & live).any()):
                raise ValueError(f'align: target ids must lie in [1, {V})')
        dev = self.device
        with torch.cuda.device(dev):
            return ctc_align_cuda(output.to(device=dev).contiguous().float(),
                                  output_len.to(device=dev, dtype=torch.int64).contiguous(), 1,
                                  targets.to(device=dev, dtype=torch.int32).contiguous(),
                                  targets_len.to(device=dev, dtype=torch.int64).contiguous())

    def error_report(self, output, output_len, val_inputs, beam_width=None):
        """PER with its breakdown: the decode of ``decode`` (same arguments; ``per`` and ``last_hyp`` are bit-identical to
        what it gives), then the Levenshtein alignment of every folded hypothesis against its folded reference:
            loss, logp, out_len = trainer.step(batch, training=False); rep = trainer.error_report(logp, out_len, batch)
        -> trainer.ErrorReport(per, counts, ref_at, hyp_at, confusion) of device tensors (see edit_align_cuda); the
        corpus substitution rate is rep.counts[:, 1].sum() / targets_len.sum().  Target ids outside [0, V) raise
        ValueError when the targets are host tensors (checked before the upload); on the device such a row comes back
        with counts -1."""
        _, (targets, targets_len) = val_inputs
        V = output.shape[2]
        if not targets.is_cuda:
            live = torch.arange(targets.shape[1])[None, :] < torch.as_tensor(targets_len).cpu()[:, None]
            if bool((((targets < 0) | (targets >= V)) & live).any()):
                raise ValueError(f'error_report: target ids must lie in [0, {V})')
        dev = self.device
        with torch.cuda.device(dev):
            per = self._decode(output, output_len, val_inputs, beam_width)
            hyp, hyp_len, _ = self.last_hyp
            ea = edit_align_cuda(hyp, hyp_len, targets.to(device=dev, dtype=torch.int32).contiguous(),
                                 targets_len.to(device=dev, dtype=torch.int64).contiguous(), self._lut, V)
        return ErrorReport(per, *ea)

    # ---------------------------------------------------------------- epoch loop (trainer.py:80-206)
    def train(self, model, epochs=40, lr=0.0001, reset=False, model_name=None):
        self.model = model
        self._model = model
        self.lr = lr
        model.to(device=self.device)
        self.optimizer = FusedAdam(model, lr=lr, eps=1e-07)
        self.scheduler = ExponentialLR(self.optimizer, 0.9)
        if self.verbose:
            print_model_summary(model)
        epoch, best_val, val_scores = 0, None, []
        latest_ckpt = best_ckpt = None
        if self.save_dir:
            d = pathlib.Path(self.save_dir)
            if model_name is not None:
                d = d / str(model_name)
            d.mkdir(exist_ok=True, parents=True)
            latest_ckpt, best_ckpt = d / 'latest.ckpt', d / 'best.ckpt'
            if best_ckpt.exists():
                if reset:
                    best_ckpt.unlink()
                else:
                    self.load(best_ckpt)
                    self.remember_best()
            if latest_ckpt.exists():
                if reset:
                    latest_ckpt.unlink()
                else:
                    self.load(latest_ckpt)
        loss_tracker, per_tracker = AvgMeter(), AvgMeter()
        warmup_limits = [1.0, 1.0, 2.0, 2.0]
        warmup = 0
        while epoch < epochs:
            set_time_limit(self.train_load, warmup_limits[warmup] if warmup < len(warmup_limits) else None)
            loss_tracker.reset()
            model.train()
            losses = []
            for batch in self.train_load:
                loss, *_ = self.step(batch, training=True)
                losses.append(loss)          # no per-batch host sync; reduce once per epoch
            for l in torch.stack(losses).tolist() if losses else []:
                loss_tracker.update(l)
            if self.verbose:
                tag = f'Warmup epoch {warmup + 1}' if warmup < len(warmup_limits) else f'Epoch {epoch + 1}'
                print(f'{tag}: average loss: {loss_tracker.get():.4f}')
            if warmup < len(warmup_limits):
                warmup += 1
                continue
            val_loss, val_per = self._evaluate(self.valid_load)
            val_scores.append((val_loss, val_per))
            if self.verbose:
                print(f'Epoch {epoch + 1}: average val loss: {val_loss:.4f}, average val per: {val_per:.4f}')
            epoch += 1
            is_best = best_val is None or val_per < best_val
            if is_best:
                best_val = val_per
                self.remember_best()
            if epoch >= 5:
                self.scheduler.step()
            if self.save_dir:
                self.save(latest_ckpt)
                if is_best:
                    self.save(best_ckpt)
        self.recall_best()
        test_loss, test_per = self._evaluate(self.test_load)
        self.model = self._model = self.lr = self.optimizer = self.scheduler = self._best_weights = None
        return val_scores, test_loss, test_per

    def _evaluate(self, loader):
        lt, pt = AvgMeter(), AvgMeter()
        self._model.eval()
        res = []
        for batch in loader:
            loss, logp, out_len = self.step(batch, training=False)
            per = self.decode(logp, out_len, batch)
            res.append(torch.stack([loss.double(), per.double()]))
        for l, p in (torch.stack(res).tolist() if res else []):
            lt.update(l)
            pt.update(p)
        return lt.get(), pt.get()

    # ---------------------------------------------------------------- checkpoints (trainer.py:249-264)
    def save(self, ckpt_name):
        torch.save({'model': {k: v.contiguous() for k, v in self._model.state_dict().items()},
                    'optim': self.optimizer.state_dict()}, str(ckpt_name))

    def load(self, ckpt_name):
        state = torch.load(str(ckpt_name), map_location=self.device)
        self._model.load_state_dict(state['model'])
        self.optimizer.load_state_dict(state['optim'])

    def remember_best(self):
        # a real copy (the reference keeps aliases of the live tensors, trainer.py:260-261)
        self._best_weights = {k: v.detach().clone() for k, v in self._model.state_dict().items()}

    def recall_best(self):
        if self._best_weights is not None:
            self._model.load_state_dict(self._best_weights)


def get_trainer(*args, **kwargs):
    return Trainer(*args, **kwargs)
