"""Plan-based executor of the candidate model on libnbasr (forward + backward + optimiser tail).

One Engine per ASRModel.  It
  * re-homes all parameters (and their .grad) into two flat fp32 buffers (the time-reduction
    conv weights are stored tap-major (C_out, k, C_in) -- the GEMM layout -- and exposed to torch
    as permuted views with the reference shape (C_out, C_in, k), so state_dict round-trips);
  * keeps bf16 operand copies (plain / transposed / tap-flipped) of the GEMM weights;
  * builds, per input shape (B, T), a static plan: zero-padded channels-last activation buffers
    and a list of C-ABI calls with pre-filled argument structs (one list for forward, one for
    backward), replayed on torch's current stream (CUDA-graph capturable: no allocation, no sync).

Forward semantics follow ASRModel.forward (model.py:116-131), SearchCell/Node (model.py:13-59),
PadConvRelu/Linear (ops.py:7-50); backward is the hand-derived adjoint (there is no autograd
inside the engine).
"""
import collections
import ctypes as C
import functools
import math
import os

import torch

from . import _lib
from ._lib import BF16, F16, F32, PAD_L, PAD_R, Epilogue, GConv, Gemm, Wgrad
from .model import CELLS_PER_BLOCK, CONV_EDGES, FEATURES, FILTERS, HIDDEN, TR_STRIDES, PadConvRelu, pad_rule

HP = 512  # padded LSTM hidden width of the h_seq buffer (TMA-friendly row pitch)
# 16-bit mode: forward activations are fp16 holding ACT_SCALE * x (a power of two keeps the rescaling exact and small
# activations out of the fp16 subnormal range; the largest representable true value is 65504 / 32 = 2047, far above
# anything a ReLU20 / LayerNorm / skip-sum net produces).  Gradients stay bf16.  See include/nbasr.h and DESIGN.md 4.
ACT_SCALE = 32.0


def _ptr(t, off_elems=0):
    return t.data_ptr() + off_elems * t.element_size()


def dense_wgrad_inputs(arch, use_norm, use_rnn, input_dropout=False):
    """Names of the forward activations that a dense (GEMM) weight gradient reads: the input of each block's time-reduction
    conv, of every `linear` edge and of the LSTM input projection (the encoder output, or its input-dropout copy).  In a
    16-bit grad plan exactly these get an unscaled bf16 twin: one tcgen05.mma cannot take the fp16 activation and the bf16
    gradient together.  The grouped-conv weight gradient needs none; it converts the fp16 tile itself (nbasr_gconv_wgrad_x).
    Names: 'input' (the transposed features), 'b{i}.ln' (block i's LayerNorm), 'b{i}.c{c}.n{n}' (node n of cell c),
    'b{i}.c{c}.ln' (cell c's LayerNorm) and 'lstm_in' (the LSTM's input dropout, only in plans with dropout)."""
    ops = [nd[0] for nd in arch]
    names = {'input'}
    for i, ncells in enumerate(CELLS_PER_BLOCK):
        cin = f'b{i}.ln'
        for c in range(ncells):
            outs = [cin] + [f'b{i}.c{c}.n{n}' for n in range(len(ops))]       # node n reads outs[n]
            names.update(outs[n] for n, op in enumerate(ops) if op == 'linear')
            cin = f'b{i}.c{c}.ln' if use_norm else outs[-1]
        if i < len(CELLS_PER_BLOCK) - 1:
            names.add(cin)
        elif use_rnn:
            names.add('lstm_in' if input_dropout else cin)
    return names


class _Geo:
    """Padded channels-last geometry of one encoder block: (B, Tp, C), frame t at row b*Tp+PAD_L+t."""

    def __init__(self, B, T, C):
        self.B, self.T, self.C = B, T, C
        tp = T + PAD_L + PAD_R
        self.Tp = tp + (tp & 1)          # even, so strided (stride-2) row views nest exactly
        self.rows = B * self.Tp + 8      # tail slack: taps may reach 8 rows past the last utterance
        self.mw = (C + 31) // 32         # mask words per row


class _Plan:
    pass


class _Arena:
    """Zero-initialised device memory for one plan, carved from a few large blocks (64 MiB, doubling up to 2 GiB): one
    fill launch per block instead of one per buffer, and everything a plan owns is freed together when it is evicted."""

    def __init__(self, dev, first_block=64 << 20):
        # first_block: an estimate of the whole arena (one fill launch, and the caching allocator hands the same block back
        # to the next plan of this shape); it only has to be roughly right -- further blocks follow the doubling rule
        self.dev, self.blocks, self.off, self.next = dev, [], 0, max(1 << 20, int(first_block))
        self.bytes = 0

    def raw(self, nbytes):
        nbytes = max(256, (nbytes + 255) & ~255)
        if not self.blocks or self.off + nbytes > self.blocks[-1].numel():
            size = max(self.next, nbytes)
            self.next = min(self.next * 2, 2 << 30)
            self.blocks.append(torch.zeros(size, dtype=torch.uint8, device=self.dev))
            self.off = 0
            self.bytes += size
        t = self.blocks[-1][self.off:self.off + nbytes]
        self.off += nbytes
        return t

    def zeros(self, shape, dtype):
        shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        n = 1
        for x in shape:
            n *= x
        nb = n * dtype.itemsize
        return self.raw(nb)[:nb].view(dtype).view(shape)


class _Mask:
    """Plane-major gate-bit mask of a (rows, C) tensor: planes of w columns, one 4/8-byte entry per row and plane."""

    def __init__(self, rows, C, w, arena):
        self.w = w
        eb = 4 if w == 32 else 8
        self.t = arena.zeros(((C + w - 1) // w) * rows * eb, torch.uint8)


def _on_device(fn):
    """Run a method with the engine's GPU as the current device: libnbasr launches on torch's CURRENT stream, so a model on
    cuda:k must not run in another device's context (Trainer(gpus=[k]) / get_model(gpu=k) without torch.cuda.set_device)."""
    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        dev = getattr(self, 'device', None)
        if dev is None:
            di = getattr(self.model, '_device_init', None)
            dev = di['device'] if di else self.params[0].device
        if dev.type != 'cuda':
            raise RuntimeError('nb_asr_b200 needs the model on a CUDA device (no CPU fallback)')
        with torch.cuda.device(dev):
            return fn(self, *a, **k)
    return wrapped


class Engine:
    def __init__(self, model, precision='bf16'):
        assert precision in ('bf16', 'fp32')
        self.model = model
        self.precision = precision
        # dt / tdt: gradients and the operands that multiply them; adt / tadt: forward activations and their weight operands
        self.dt = BF16 if precision == 'bf16' else F32
        self.tdt = torch.bfloat16 if precision == 'bf16' else torch.float32
        self.adt = F16 if precision == 'bf16' else F32
        self.tadt = torch.float16 if precision == 'bf16' else torch.float32
        self.S = ACT_SCALE if precision == 'bf16' else 1.0
        self.lib = _lib.load()
        self.params = list(model.parameters())
        self.names = [n for n, _ in model.named_parameters()]
        self.plans = collections.OrderedDict()      # (B, T, training) -> plan, least recently used first
        self.max_plans = int(os.environ.get('NBASR_MAX_PLANS', '6'))
        self.device = None
        self.flat_p = None
        self._pack_version = None
        self._bound_ptr = None
        self.training_drop = float(model.dropout_rate)
        self.launches = 0

    # ------------------------------------------------------------------ parameter binding
    def _is_dense_conv_w(self, name):
        return name.endswith('.conv.weight') and name.count('.') == 3   # model.{i}.conv.weight

    def bind(self):
        p0 = self.params[0]
        if self.flat_p is not None and self._bound_ptr == (p0.data_ptr(), p0.device):
            return
        dinit = getattr(self.model, '_device_init', None)
        dev = dinit['device'] if dinit else p0.device
        if dev.type != 'cuda':
            raise RuntimeError('nb_asr_b200 needs the model on a CUDA device (no CPU fallback)')
        with torch.cuda.device(dev):
            self._bind(dev)

    def _bind(self, dev):
        # a re-bind (model.to(other device), load_state_dict(assign=True), ...) keeps the optimiser state
        old = (self.adam_m, self.adam_v, self.opt_state) if self.flat_p is not None else None
        self.device = dev
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 63) // 64 * 64
        flat_p = torch.zeros(total, dtype=torch.float32, device=dev)
        flat_g = torch.zeros(total, dtype=torch.float32, device=dev)
        self.slices = {}
        dinit = getattr(self.model, '_device_init', None)       # get_model(init='device'): parameters have no storage yet
        gen = torch.Generator(device=dev).manual_seed(dinit['seed']) if dinit else None
        with torch.no_grad():
            for i, (name, p, off) in enumerate(zip(self.names, self.params, offs)):
                n = p.numel()
                dst, gdst = flat_p[off:off + n], flat_g[off:off + n]
                if self._is_dense_conv_w(name):
                    co, ci, k = p.shape
                    pv, gv = dst.view(co, k, ci).permute(0, 2, 1), gdst.view(co, k, ci).permute(0, 2, 1)
                else:
                    pv, gv = dst.view(p.shape), gdst.view(p.shape)
                if dinit:
                    # storage-less (meta) parameter: draw the values on the device, then swap in a real Parameter that views
                    # the flat buffer (a meta tensor cannot be re-pointed with .data)
                    self._device_init_param(name, p, dst, gen, dinit['conv_gain'])
                    newp = torch.nn.Parameter(pv, requires_grad=p.requires_grad)
                    mod_name, _, leaf = name.rpartition('.')
                    self.model.get_submodule(mod_name)._parameters[leaf] = newp
                    self.params[i] = p = newp
                else:
                    pv.copy_(p.detach().to(dev))
                    p.data = pv
                p.grad = gv
                self.slices[name] = (off, n)
        if dinit:
            self.model._device_init = None       # a later re-bind copies the (now real) parameters like any other
        self.flat_p, self.flat_g = flat_p, flat_g
        self.n_flat = total
        self.adam_m = torch.zeros_like(flat_p)
        self.adam_v = torch.zeros_like(flat_p)
        if old is not None and old[0].numel() == total:
            self.adam_m.copy_(old[0])
            self.adam_v.copy_(old[1])
        reg = [self.slices[n] for n in self.names if n.endswith('.conv.weight')]
        self.seg_off = torch.tensor([o for o, _ in reg], dtype=torch.int64, device=dev)
        self.seg_len = torch.tensor([l for _, l in reg], dtype=torch.int64, device=dev)
        self.seg_chunks = int(sum((l + 16383) // 16384 for _, l in reg))
        # [step, lr, ||g||^2, clip, per-segment ||W||^2 ...] + scratch of the deterministic reductions (nbasr.h)
        self.opt_state = torch.zeros(8 + len(reg) + 592 + self.seg_chunks, dtype=torch.float32, device=dev)
        if old is not None and old[2].numel() == self.opt_state.numel():
            self.opt_state.copy_(old[2])
        self._lr_host = None          # the device copy of lr is rewritten by the next set_lr()
        self.drop_step = torch.zeros(1, dtype=torch.int64, device=dev)
        self._bound_ptr = (self.params[0].data_ptr(), dev)
        self.seg_chunks = int(sum((l + 16383) // 16384 for _, l in reg))
        self._build_packs()
        self._compile_pack_jobs()
        self.plans = collections.OrderedDict()
        self._pack_version = None

    @staticmethod
    def _device_init_param(name, p, dst, gen, conv_gain):
        """model/torch/__init__.py:13-29 on the device: xavier_uniform for Linear / Conv1d / LSTM weights (torch's fan
        rule: fan_in = size(1) * receptive field, fan_out = size(0) * receptive field), zeros for biases, LayerNorm (1, 0).
        i.i.d. entries: the tap-major storage of the dense conv weights needs no permutation."""
        leaf = name.rsplit('.', 1)[-1]
        if p.dim() >= 2:
            rf = 1
            for d in p.shape[2:]:
                rf *= d
            bound = math.sqrt(6.0 / (p.shape[1] * rf + p.shape[0] * rf))
            if '.nodes.' in name and name.endswith('.conv.weight'):
                bound *= conv_gain
            dst.uniform_(-bound, bound, generator=gen)
        elif leaf == 'weight':            # LayerNorm gamma
            dst.fill_(1.0)
        else:
            dst.zero_()

    def P(self, name):
        off, _ = self.slices[name]
        return self.flat_p.data_ptr() + 4 * off

    def G(self, name):
        off, _ = self.slices[name]
        return self.flat_g.data_ptr() + 4 * off

    # ------------------------------------------------------------------ operand copies
    def _build_packs(self):
        """Describe every derived weight buffer; (re)filled by refresh_packs()."""
        m = self.model
        dev, tdt, tadt, adt = self.device, self.tdt, self.tadt, self.adt
        # wf: FORWARD operands (multiply activations: activation format, fp16 in 16-bit mode);
        # wd / wt: INPUT-GRADIENT operands (multiply gradients: bf16 in 16-bit mode)
        parena = self.pack_arena = _Arena(dev)      # every derived operand lives in one zero-filled arena
        self.pack_ops = []     # (cfunc, args) without stream
        self.wf, self.wd, self.wt = {}, {}, {}
        lib = self.lib
        idx = 0
        self.block_conv, self.block_ln, self.block_cells = [], [], []
        for i in range(4):
            cin = FEATURES if i == 0 else FILTERS[i - 1]
            cout = FILTERS[i]
            name = f'model.{idx}.conv'
            self.block_conv.append(name)
            n = cout * 8 * cin
            if self.dt == BF16:
                buf = parena.zeros(n, tadt)
                self.pack_ops.append((lib.nbasr_convert, (self.P(name + '.weight'), buf.data_ptr(), adt, n)))
                self.wf[name] = buf
            else:
                self.wf[name] = None   # flat fp32 master is already (C_out, 8*C_in)
            if i > 0:
                if TR_STRIDES[i] == 1:
                    specs = [(8, 7, -1)]
                else:
                    specs = [(4, 7, -2), (4, 6, -2)]
                bufs = []
                for nq, t0, ts in specs:
                    b = parena.zeros(cin * nq * cout, tdt)
                    # out[n=ci][q*Cout + co] = w[co][t0+q*ts][ci]
                    self.pack_ops.append((lib.nbasr_pack_weight, (self.P(name + '.weight'), b.data_ptr(), self.dt, cout, cin,
                                                                   nq, t0, ts, 8 * cin, 1, cin)))
                    bufs.append(b)
                self.wd[name] = bufs
            idx += 1
            self.block_ln.append(f'model.{idx}')
            idx += 1
            cells = []
            for _ in range(CELLS_PER_BLOCK[i]):
                cells.append(f'model.{idx}')
                for nn_, node in enumerate(m.arch_desc):
                    op = node[0]
                    pn = f'model.{idx}.nodes.{nn_}.op'
                    if op == 'linear':
                        n = cout * cout
                        if self.dt == BF16:
                            b = parena.zeros(n, tadt)
                            self.pack_ops.append((lib.nbasr_convert, (self.P(pn + '.linear.weight'), b.data_ptr(), adt, n)))
                            self.wf[pn] = b
                        else:
                            self.wf[pn] = None
                        bt = parena.zeros(n, tdt)
                        self.pack_ops.append((lib.nbasr_pack_weight, (self.P(pn + '.linear.weight'), bt.data_ptr(), self.dt,
                                                                       cout, cout, 1, 0, 0, cout, 1, 0)))
                        self.wt[pn] = bt
                    elif op in CONV_EDGES:
                        k, _ = CONV_EDGES[op]
                        cpg = cout // 100
                        if self.dt == BF16:
                            # block-diagonal bf16 operands of the tcgen05 grouped-conv kernel (forward / input-gradient)
                            ne = int(lib.nbasr_gconv_mma_pack_elems(cout, cpg, k))
                            # zeros: the batched refresh only rewrites the diagonal blocks (pack_batch.cu kind 2)
                            bf_, bt = parena.zeros(ne, tadt), parena.zeros(ne, tdt)
                            for buf, odt, tr_ in ((bf_, adt, 0), (bt, BF16, 1)):
                                self.pack_ops.append((lib.nbasr_pack_gconv_mma, (self.P(pn + '.conv.weight'), buf.data_ptr(), odt, cout, cpg, k, tr_)))
                            self.wf[pn] = bf_
                        else:
                            bt = parena.zeros(cout * cpg * k, torch.float32)
                            self.pack_ops.append((lib.nbasr_pack_gconv_dgrad, (self.P(pn + '.conv.weight'), bt.data_ptr(), cout, cpg, k)))
                        self.wt[pn] = bt
                idx += 1
            self.block_cells.append(cells)
        if m.use_rnn:
            idx += 1
            self.lstm_name = f'model.{idx}'
            ln = self.lstm_name
            n = 4 * HIDDEN * FILTERS[-1]
            if self.dt == BF16:
                b = parena.zeros(n, tadt)
                self.pack_ops.append((lib.nbasr_convert, (self.P(ln + '.weight_ih_l0'), b.data_ptr(), adt, n)))
                self.wf[ln] = b
            else:
                self.wf[ln] = None
            bt = parena.zeros(n, tdt)
            self.pack_ops.append((lib.nbasr_pack_weight, (self.P(ln + '.weight_ih_l0'), bt.data_ptr(), self.dt, 4 * HIDDEN,
                                                           FILTERS[-1], 1, 0, 0, FILTERS[-1], 1, 0)))
            self.wt[ln] = bt
            self.lstm_bias = parena.zeros(4 * HIDDEN, torch.float32)
            self.whh_packed = None
            if self.dt == BF16:
                # W_hh operand of the tcgen05 cluster recurrence: [16 CTAs][gate*32 + unit][512] bf16
                self.whh_packed = parena.zeros(16 * 128 * 512, tdt)
                self.pack_ops.append(('lstm_whh', (self.P(ln + '.weight_hh_l0'), self.whh_packed.data_ptr(), HIDDEN)))
            idx += 1
        self.head_name = f'model.{idx}'

    def _compile_pack_jobs(self):
        """Translate the per-buffer pack calls into one device-resident job table (single launch per refresh)."""
        import ctypes as C_
        lib = self.lib
        kinds = {'nbasr_convert': 0, 'nbasr_pack_weight': 1, 'nbasr_pack_gconv_mma': 2, 'nbasr_pack_gconv_dgrad': 3}
        jobs = (_lib.PackJob * len(self.pack_ops))()
        blocks = 0
        for j, (fn, a) in zip(jobs, self.pack_ops):
            if fn == 'lstm_whh':
                j.kind, j.src, j.dst, j.out_dtype, j.n_out = 4, a[0], a[1], BF16, 16 * 128 * 512
                j.a[0] = a[2]
                blocks += self._pack_chunks(j)
                continue
            j.kind = kinds[fn.__name__]
            if j.kind == 0:
                src, dst, odt, n = a
                j.src, j.dst, j.out_dtype, j.n_out = src, dst, odt, n
            elif j.kind == 1:
                src, dst, odt, M, N, nq, t0, ts, wm, wn, wt = a
                j.src, j.dst, j.out_dtype, j.n_out = src, dst, odt, N * nq * M
                j.a[0], j.a[1], j.a[2], j.a[3], j.a[4] = M, N, nq, t0, ts
                j.s[0], j.s[1], j.s[2] = wm, wn, wt
            elif j.kind == 2:
                src, dst, odt, Cc, cpg, k, tr_ = a
                j.src, j.dst, j.out_dtype = src, dst, odt
                j.n_out = int(lib.nbasr_gconv_mma_pack_elems(Cc, cpg, k))
                j.a[0], j.a[1], j.a[2], j.a[3] = Cc, cpg, k, tr_
            else:
                src, dst, Cc, cpg, k = a
                j.src, j.dst, j.out_dtype, j.n_out = src, dst, F32, Cc * cpg * k
                j.a[0], j.a[1], j.a[2] = Cc, cpg, k
            blocks += self._pack_chunks(j)
        raw = bytes(jobs)
        self.pack_jobs = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.device)
        bmap = []
        for ji, j in enumerate(jobs):
            nch = self._pack_chunks(j)
            bmap.append(torch.stack([torch.full((nch,), ji, dtype=torch.int32), torch.arange(nch, dtype=torch.int32)], 1))
        self.pack_blockmap = torch.cat(bmap).contiguous().to(self.device)
        self.pack_njobs, self.pack_blocks = len(self.pack_ops), blocks

    @staticmethod
    def _pack_chunks(j):
        """blocks of one pack job: 64x64 transpose tiles per tap for kind 1, 4096-element chunks otherwise"""
        if j.kind == 1:
            M, N, nq = j.a[0], j.a[1], j.a[2]
            return nq * ((M + 63) // 64) * ((N + 63) // 64)
        if j.kind == 2:
            return (j.a[0] * j.a[1] * j.a[2] + 4095) // 4096      # walks the source weights (C * cpg * ktaps)
        return (j.n_out + 4095) // 4096

    def _param_version(self):
        return sum(p._version for p in self.params)

    @_on_device
    def refresh_packs(self, force=False):
        v = self._param_version()
        if not force and v == self._pack_version:
            return
        st = torch.cuda.current_stream().cuda_stream
        if self.pack_njobs:
            _lib.check(self.lib.nbasr_pack_batch(self.pack_jobs.data_ptr(), self.pack_njobs, self.pack_blockmap.data_ptr(), self.pack_blocks, st), 'pack_batch')
            self.launches += 1
        if self.model.use_rnn:
            off_i, n = self.slices[self.lstm_name + '.bias_ih_l0']
            off_h, _ = self.slices[self.lstm_name + '.bias_hh_l0']
            torch.add(self.flat_p[off_i:off_i + n], self.flat_p[off_h:off_h + n], out=self.lstm_bias)
        self._pack_version = v

    # ------------------------------------------------------------------ plan construction
    def _epi(self, ld, bias=0, relu=0, drop_p=0.0, salt=0, adds=(), out=0, out_dtype=None, mask_out=None, out2=0,
             mask2=None, scale2=1.0, mask_rows=0, accumulate=0, fwd=False, copy=0, acc_scale=1.0):
        """mask_out / mask2 are _Mask objects (tensor + plane width) or None.
        fwd=True: a FORWARD epilogue in the scaled activation domain (16-bit mode: fp16 tensors holding S*x): bias and the
        ReLU20 bound are scaled by S, skip tensors and `out` are activation-format; copy = optional unscaled bf16 copy of
        `out` for the weight gradient that will read this tensor (out2 slot, scale 1/S)."""
        e = Epilogue()
        if fwd:
            e.acc_scale, e.bias_scale, e.relu_hi = acc_scale, self.S, 20.0 * self.S
            act = self.adt
            if copy:
                assert not out2
                out2, scale2, mask2 = copy, 1.0 / self.S, None
        else:
            e.acc_scale, e.bias_scale, e.relu_hi = acc_scale, 1.0, 20.0
            act = self.dt
        e.bias = bias or None
        e.relu20 = relu
        e.drop_p = drop_p
        e.drop_seed = salt
        e.drop_step = self.drop_step.data_ptr() if drop_p > 0 else None
        e.n_add = len(adds)
        for i, a in enumerate(adds):
            e.add[i] = a
        e.add_dtype = act
        e.out = out or None
        e.out_dtype = act if out_dtype is None else out_dtype
        e.ld_out = ld
        e.mask_out = mask_out.t.data_ptr() if mask_out is not None else None
        e.mask_w = mask_out.w if mask_out is not None else 32
        e.out2 = out2 or None
        e.out2_dtype = self.dt
        e.mask2 = mask2.t.data_ptr() if mask2 is not None else None
        e.mask2_w = mask2.w if mask2 is not None else 32
        e.scale2 = scale2
        e.mask_rows = mask_rows
        e.accumulate = accumulate
        return e

    def plan(self, B, T, training, grad=None, input_grad=False):
        """Plans are cached per (B, T, training, grad[, 'input_grad']), least recently used first.  `training` switches
        dropout on; `grad` (default: training) says whether a backward pass may follow: only then are gate-bit masks, bf16
        twins of the forward activations a dense weight gradient reads and the backward call list built (an eval step needs none of them).  `input_grad`
        (implies grad) appends the gradient wrt the input features to the backward pass: pl.daudio (B, 80, T) fp32.  A plan
        owns every activation / mask / gradient buffer of its shape (at 64 x 500 on the default arch: 4.6 GB for a grad plan, 3.0 GB for an eval plan) plus the CUDA graphs and CTC workspaces captured on it, so
        loaders whose padded length changes from batch to batch would otherwise grow without bound: beyond `max_plans`
        (NBASR_MAX_PLANS, default 6) the oldest plan is dropped and its memory returns to the allocator."""
        grad = bool(training) if grad is None else bool(grad)
        input_grad = bool(input_grad)
        grad = grad or input_grad
        key = (B, T, bool(training), grad) + (('input_grad',) if input_grad else ())
        pl = self.plans.get(key)
        if pl is None:
            while len(self.plans) >= max(1, self.max_plans):
                _, old = self.plans.popitem(last=False)
                old.graphs.clear()
                old.ws.clear()
            pl = self.plans[key] = self._build_plan(B, T, bool(training), grad, input_grad)
        else:
            self.plans.move_to_end(key)
        return pl

    def _plan_bytes_estimate(self, B, T, grad):
        """Rough size of a plan's arena: per encoder block (2 + 4 per cell) activation buffers, with gradients also the
        bf16 twins of those a dense weight gradient reads, 7 gradient buffers and 1 bit per element of gate masks; head and
        small buffers on top."""
        es = 2 if self.dt == BF16 else 4
        twins = dense_wgrad_inputs(self.model.arch_desc, self.model.use_norm, self.model.use_rnn) if self.adt != self.dt else ()
        total, Tcur = B * (T + 16) * FEATURES * es * 2, T
        for i in range(4):
            Tcur = Tcur if TR_STRIDES[i] == 1 else (Tcur + 1) // 2
            rows = B * (Tcur + PAD_L + PAD_R + 1) + 8
            per = rows * FILTERS[i] * es
            nbuf = 2 + 4 * CELLS_PER_BLOCK[i]
            total += per * nbuf
            if grad:
                ntw = sum(1 for n in twins if n.startswith(f'b{i}.'))
                total += per * (ntw + 7) + per * nbuf // (8 * es) + per // 4
        total += B * Tcur * (4 * HIDDEN * 4 * (3 if grad else 1) + HP * 2 + HIDDEN * 4 * 3 + 49 * 4 * 3)
        return int(total * 1.05) + (8 << 20)

    @_on_device
    def _build_plan(self, B, T, training, grad=True, input_grad=False):
        self.bind()
        m, lib, dev, dt, tdt = self.model, self.lib, self.device, self.dt, self.tdt
        es = 2 if dt == BF16 else 4
        pl = _Plan()
        pl.B, pl.T, pl.training, pl.grad, pl.input_grad = B, T, training, grad, input_grad
        pl.keep = []       # keeps ctypes structs / tensors alive
        pl.graphs, pl.ws = {}, {}     # CUDA graphs / CTC workspaces captured on this plan (trainer.py); die with the plan
        arena = pl.arena = _Arena(dev, self._plan_bytes_estimate(B, T, grad))
        fwd, bwd_rev = [], []   # bwd_rev: groups appended in forward order, executed reversed
        drop_p = self.training_drop if training else 0.0
        dscale = 1.0 / (1.0 - drop_p) if drop_p > 0 else 1.0
        salt = [1]

        def next_salt():
            salt[0] += 1
            return salt[0] * 0x9E3779B1

        adt, tadt, S = self.adt, self.tadt, self.S
        twin_plan = grad and adt != dt
        twin_names = dense_wgrad_inputs(m.arch_desc, m.use_norm, m.use_rnn, input_dropout=drop_p > 0) if twin_plan else ()
        bcopy = {}          # id(forward activation) -> its unscaled bf16 twin (grad plans of the 16-bit mode)
        pl.twins = {}       # activation name -> bf16 twin

        def zbuf(rows, cols, dtype=None):
            return arena.zeros((rows, cols), tdt if dtype is None else dtype)

        def zact(rows, cols, name=None):
            """forward activation buffer (activation format) and, if a dense weight gradient reads it in a 16-bit grad
            plan, its bf16 twin"""
            t = arena.zeros((rows, cols), tadt)
            if name in twin_names:
                bcopy[id(t)] = pl.twins[name] = arena.zeros((rows, cols), tdt)
            return t

        def Bc(t):
            """the tensor a dense weight gradient reads for forward activation t"""
            return bcopy[id(t)] if twin_plan else t

        def cptr(t):
            c = bcopy.get(id(t))
            return c.data_ptr() if c is not None else 0

        def call(lst, fn, *args):
            pl.keep.append(args)
            lst.append((fn, args))

        def gemm(lst, a_ptr, a_bs, a_rs, nb, nr, K, N, w_ptr, ldw, o_r0, o_bs, o_rs, epi, dtype=None):
            g = Gemm()
            g.dtype = dt if dtype is None else dtype
            g.a, g.a_bs, g.a_rs, g.nb, g.nr, g.K, g.N = a_ptr, a_bs, a_rs, nb, nr, K, N
            g.w, g.ldw, g.o_r0, g.o_bs, g.o_rs, g.epi = w_ptr, ldw, o_r0, o_bs, o_rs, epi
            call(lst, lib.nbasr_gemm_tn, C.byref(g))
            pl.keep.append(g)

        def wgrad(lst, dy_ptr, dy_bs, dy_rs, x_ptr, x_bs, x_rs, nb, nr, M, N, dw_ptr, ldw, dtype=None, dbias=None):
            w = Wgrad()
            w.dbias = dbias
            w.dtype = dt if dtype is None else dtype
            w.dy, w.dy_bs, w.dy_rs, w.x, w.x_bs, w.x_rs = dy_ptr, dy_bs, dy_rs, x_ptr, x_bs, x_rs
            w.nb, w.nr, w.M, w.N, w.dw, w.ldw = nb, nr, M, N, dw_ptr, ldw
            call(lst, lib.nbasr_gemm_wgrad, C.byref(w))
            pl.keep.append(w)

        # ---- input
        pl.audio = arena.zeros((B, FEATURES, T), torch.float32)
        g_in = _Geo(B, T, FEATURES)
        x_in = zact(g_in.rows, FEATURES, 'input')
        call(fwd, lib.nbasr_transpose_in, pl.audio.data_ptr(), x_in.data_ptr(), adt, B, FEATURES, T, g_in.Tp, S)
        if cptr(x_in):
            call(fwd, lib.nbasr_transpose_in, pl.audio.data_ptr(), cptr(x_in), dt, B, FEATURES, T, g_in.Tp, 1.0)

        prev, pg = x_in, g_in
        Tcur = T
        arch = m.arch_desc
        pl.block_geo = []
        # ReLU20 layers of a grad plan in forward order, (gate mask, block geometry, block index): what the NASWOT proxy
        # reads (proxies.nwot_kernel).  The block convs' and the non-`zero` node ops' masks; nothing else carries one.
        pl.gates = [] if grad else None
        # backward bookkeeping: per block a pool of gradient buffers
        gpools = []
        block_records = []
        for i in range(4):
            s = TR_STRIDES[i]
            Ti = Tcur if s == 1 else (Tcur + 1) // 2
            geo = _Geo(B, Ti, FILTERS[i])
            pl.block_geo.append(geo)
            Cc, Tp, mw = geo.C, geo.Tp, geo.mw
            cname = self.block_conv[i]
            lpad, _ = pad_rule(8, 1, s)
            K = 8 * pg.C
            z = zact(geo.rows, Cc)
            zmask = _Mask(geo.rows, Cc, 32, arena) if grad else None     # gate bits are only read by the backward pass
            pl.keep.append(zmask)
            if grad:
                pl.gates.append((zmask, geo, i))
            wf_ptr = self.wf[cname].data_ptr() if self.wf[cname] is not None else self.P(cname + '.weight')
            a_ptr = _ptr(prev, (PAD_L - lpad) * pg.C)
            a_ptr_b = _ptr(Bc(prev), (PAD_L - lpad) * pg.C)      # the same rows of the bf16 copy (weight gradient)
            epi = self._epi(Cc, bias=self.P(cname + '.bias'), relu=1, out=z.data_ptr(), mask_out=zmask, mask_rows=geo.rows, fwd=True)
            gemm(fwd, a_ptr, pg.Tp * pg.C, s * pg.C, B, Ti, K, Cc, wf_ptr, K, PAD_L, Tp, 1, epi, dtype=adt)
            y = zact(geo.rows, Cc, f'b{i}.ln')
            mean0 = zbuf(geo.rows, 1, torch.float32)
            rstd0 = zbuf(geo.rows, 1, torch.float32)
            lname = self.block_ln[i]
            # scaled fp16 input S*x: eps*S^2 gives the exact xhat of the unscaled tensor; output again scaled by S
            call(fwd, lib.nbasr_layernorm_fwd, adt, z.data_ptr(), y.data_ptr(), B, Ti, Tp, Cc, self.P(lname + '.weight'),
                 self.P(lname + '.bias'), 1e-3 * S * S, mean0.data_ptr(), rstd0.data_ptr(), S, cptr(y) or None)
            rec = dict(i=i, geo=geo, prev=prev, pg=pg, z=z, zmask=zmask, y=y, mean=mean0, rstd=rstd0, cells=[],
                       a_ptr=a_ptr_b, K=K, s=s, lpad=lpad)
            cur = y
            for ci, cellname in enumerate(self.block_cells[i]):
                outs = [cur]
                crec = dict(name=cellname, outs=outs, masks=[], nodes=[])
                for n, node in enumerate(arch):
                    op, branches = node[0], node[1:]
                    src = outs[-1]
                    skips = [outs[k] for k, bit in enumerate(branches) if bit]
                    o = zact(geo.rows, Cc, f'b{i}.c{ci}.n{n}')
                    pn = f'{cellname}.nodes.{n}.op'
                    nrec = dict(op=op, branches=list(branches), pn=pn, mask=None, salt=0)
                    adds = [t.data_ptr() for t in skips]
                    if op == 'zero':
                        epi = self._epi(Cc, adds=adds, out=o.data_ptr(), fwd=True, copy=cptr(o))
                        call(fwd, lib.nbasr_eltwise, adt, None, Cc, B, Ti, Tp, Cc, C.byref(epi))
                        pl.keep.append(epi)
                    else:
                        # plane width = the producing kernel's slab: 32 (GEMM / SIMT) or 48/40 (tcgen05 grouped conv)
                        mwid = (40 if Cc // 100 == 10 else 48) if (op in CONV_EDGES and dt == BF16) else 32
                        mask = _Mask(geo.rows, Cc, mwid, arena) if grad else None
                        pl.keep.append(mask)
                        nrec['mask'] = mask
                        if grad:
                            pl.gates.append((mask, geo, i))
                        sl = next_salt()
                        if op == 'linear':
                            epi = self._epi(Cc, bias=self.P(pn + '.linear.bias'), relu=1, drop_p=drop_p, salt=sl, adds=adds,
                                            out=o.data_ptr(), mask_out=mask, mask_rows=geo.rows, fwd=True, copy=cptr(o))
                            w_ptr = self.wf[pn].data_ptr() if self.wf[pn] is not None else self.P(pn + '.linear.weight')
                            gemm(fwd, _ptr(src, PAD_L * Cc), Tp * Cc, Cc, B, Ti, Cc, Cc, w_ptr, Cc, PAD_L, Tp, 1, epi, dtype=adt)
                        else:
                            k, d = CONV_EDGES[op]
                            lp, _ = pad_rule(k, d, 1)
                            gc = GConv()
                            gc.dtype, gc.x, gc.B, gc.T, gc.Tp, gc.C, gc.cpg = adt, src.data_ptr(), B, Ti, Tp, Cc, Cc // 100
                            gc.ktaps, gc.off0, gc.dstep = k, -lp, d
                            if dt == BF16:
                                gc.w, gc.w_packed = self.wf[pn].data_ptr(), 3     # packed | stable (re-packed by the optimiser tail)
                            else:
                                gc.w, gc.w_packed = self.P(pn + '.conv.weight'), 0
                            gc.epi = self._epi(Cc, bias=self.P(pn + '.conv.bias'), relu=1, drop_p=drop_p, salt=sl, adds=adds,
                                               out=o.data_ptr(), mask_out=mask, mask_rows=geo.rows, fwd=True, copy=cptr(o))
                            call(fwd, lib.nbasr_gconv_fwd, C.byref(gc))
                            pl.keep.append(gc)
                            nrec.update(k=k, d=d, lp=lp)
                    crec['nodes'].append(nrec)
                    outs.append(o)
                if m.use_norm:
                    co = zact(geo.rows, Cc, f'b{i}.c{ci}.ln')
                    mean = zbuf(geo.rows, 1, torch.float32)
                    rstd = zbuf(geo.rows, 1, torch.float32)
                    call(fwd, lib.nbasr_layernorm_fwd, adt, outs[-1].data_ptr(), co.data_ptr(), B, Ti, Tp, Cc,
                         self.P(cellname + '.norm_layer.weight'), self.P(cellname + '.norm_layer.bias'), 1e-3 * S * S,
                         mean.data_ptr(), rstd.data_ptr(), S, cptr(co) or None)
                    crec.update(mean=mean, rstd=rstd, out=co)
                    cur = co
                else:
                    crec.update(out=outs[-1])
                    cur = outs[-1]
                rec['cells'].append(crec)
            block_records.append(rec)
            prev, pg, Tcur = cur, geo, Ti

        # ---- head
        geo3 = pl.block_geo[-1]
        Tq, Tp3, C3 = geo3.T, geo3.Tp, geo3.C
        pl.Tq = Tq
        V = m.num_classes + 1
        pl.V = V
        pl.logits = arena.zeros((B, Tq, V), torch.float32)
        pl.logp = arena.zeros((B, Tq, V), torch.float32)
        hn = self.head_name
        head = dict()
        if m.use_rnn:
            ln = self.lstm_name
            if drop_p > 0:
                lin = zact(geo3.rows, C3, 'lstm_in')
                dmask = _Mask(geo3.rows, C3, 32, arena)
                pl.keep.append(dmask)
                epi = self._epi(C3, drop_p=drop_p, salt=next_salt(), out=lin.data_ptr(), mask_out=dmask, mask_rows=geo3.rows,
                                fwd=True, copy=cptr(lin))
                call(fwd, lib.nbasr_eltwise, adt, prev.data_ptr(), C3, B, Tq, Tp3, C3, C.byref(epi))
                pl.keep.append(epi)
            else:
                lin, dmask = prev, None
            H4 = 4 * HIDDEN
            gx = zbuf(B * Tq, H4, torch.float32)
            wih = self.wf[ln].data_ptr() if self.wf[ln] is not None else self.P(ln + '.weight_ih_l0')
            # the LSTM wants true values: un-scale the accumulator of the scaled fp16 operand
            epi = self._epi(H4, bias=self.lstm_bias.data_ptr(), out=gx.data_ptr(), out_dtype=F32, acc_scale=1.0 / S)
            gemm(fwd, _ptr(lin, PAD_L * C3), Tp3 * C3, C3, B, Tq, C3, H4, wih, C3, 0, Tq, 1, epi, dtype=adt)
            gh = _Geo(B, Tq, HP)
            hseq = zbuf(gh.rows, HP)
            gates = zbuf(B * Tq, H4, torch.float32)
            cst = zbuf(B * Tq, HIDDEN, torch.float32)
            work = zbuf(1, 2 * B * HIDDEN + 256, torch.float32)
            call(fwd, lib.nbasr_lstm_fwd, gx.data_ptr(), self.P(ln + '.weight_hh_l0'), Tq, B, HIDDEN, _ptr(hseq, PAD_L * HP), dt,
                 gh.Tp * HP, HP, HP, gates.data_ptr(), cst.data_ptr(),
                 self.whh_packed.data_ptr() if self.whh_packed is not None else None, work.data_ptr())
            call(fwd, lib.nbasr_head_fwd, dt, _ptr(hseq, PAD_L * HP), gh.Tp * HP, HP, B, Tq, HIDDEN, V, self.P(hn + '.weight'),
                 self.P(hn + '.bias'), pl.logits.data_ptr(), pl.logp.data_ptr())
            head.update(lin=lin, dmask=dmask, gx=gx, hseq=hseq, gh=gh, gates=gates, cst=cst, work=work)
        else:
            hsrc = prev
            if adt != dt:
                # the classifier kernels read bf16 / fp32: un-scale the fp16 encoder output once
                hsrc = zbuf(geo3.rows, C3)
                epi = self._epi(C3, out=hsrc.data_ptr(), acc_scale=1.0 / S)
                call(fwd, lib.nbasr_eltwise, adt, prev.data_ptr(), C3, B, Tq, Tp3, C3, C.byref(epi))
                pl.keep.append(epi)
            head.update(hsrc=hsrc)
            call(fwd, lib.nbasr_head_fwd, dt, _ptr(hsrc, PAD_L * C3), Tp3 * C3, C3, B, Tq, C3, V, self.P(hn + '.weight'),
                 self.P(hn + '.bias'), pl.logits.data_ptr(), pl.logp.data_ptr())
        pl.fwd = fwd
        pl.final = prev
        if not grad:
            pl.bwd, pl.buckets = None, []
            return pl

        # =========================================================== backward plan
        bwd = []
        pl.dlogits = arena.zeros((B, Tq, V), torch.float32)
        # gradient wrt the last cell output of block 3 (act dtype, padded geometry)
        pools = []
        for geo in pl.block_geo:
            pools.append([zbuf(geo.rows, geo.C) for _ in range(5)])
        # one dZ buffer per node: the weight gradients of a cell's consecutive conv nodes run after all of their input
        # gradients and read every node's dZ
        dzs = [[zbuf(geo.rows, geo.C) for _ in range(max(2, len(arch)))] for geo in pl.block_geo]

        gout = pools[3].pop()
        if m.use_rnn:
            ln = self.lstm_name
            H4 = 4 * HIDDEN
            dh = zbuf(B * Tq, HIDDEN, torch.float32)
            if dt == BF16:
                # dh on CUDA cores (fp32 W), dW / db on the tensor cores from a bf16 copy of dlogits and the bf16 h_seq
                dl16 = zbuf(B * Tq, 64)
                call(bwd, lib.nbasr_head_bwd_dh, B, Tq, HIDDEN, V, self.P(hn + '.weight'), pl.dlogits.data_ptr(), dh.data_ptr(),
                     Tq * HIDDEN, HIDDEN, dl16.data_ptr())
                wgrad(bwd, dl16.data_ptr(), Tq * 64, 64, _ptr(head['hseq'], PAD_L * HP), head['gh'].Tp * HP, HP, B, Tq, V, HIDDEN,
                      self.G(hn + '.weight'), HIDDEN, dbias=self.G(hn + '.bias'))
            else:
                call(bwd, lib.nbasr_head_bwd, dt, _ptr(head['hseq'], PAD_L * HP), head['gh'].Tp * HP, HP, B, Tq, HIDDEN, V,
                     self.P(hn + '.weight'), pl.dlogits.data_ptr(), dh.data_ptr(), Tq * HIDDEN, HIDDEN, self.G(hn + '.weight'),
                     self.G(hn + '.bias'))
            dgx = zbuf(B * Tq, H4, torch.float32)
            dgx_a = zbuf(B * Tq, H4) if dt == BF16 else dgx     # bf16 copy written by the cluster kernel itself
            call(bwd, lib.nbasr_lstm_bwd, dh.data_ptr(), Tq * HIDDEN, HIDDEN, HIDDEN, self.P(ln + '.weight_hh_l0'),
                 head['gates'].data_ptr(), head['cst'].data_ptr(), Tq, B, HIDDEN, dgx.data_ptr(), head['work'].data_ptr(),
                 self.whh_packed.data_ptr() if self.whh_packed is not None else None,
                 dgx_a.data_ptr() if dt == BF16 else None)
            # biases: column sums of dgx (B*Tq rows, unpadded) -> both bias vectors.  bf16: fused into the two tensor-core
            # weight-gradient GEMMs below (ones operand, like the conv / linear bias gradients); fp32: column-sum kernel
            fuse_b = dt == BF16
            if not fuse_b:
                for bn in ('.bias_ih_l0', '.bias_hh_l0'):
                    call(bwd, lib.nbasr_colsum, F32, dgx.data_ptr() - PAD_L * H4 * 4, 1, B * Tq, B * Tq, H4, self.G(ln + bn))
            # dW_ih += dgx^T X ; dW_hh += dgx^T H_{t-1} (h_seq shifted one row up; row -1 is a zero pad row)
            wgrad(bwd, dgx_a.data_ptr(), Tq * H4, H4, _ptr(Bc(head['lin']), PAD_L * C3), Tp3 * C3, C3, B, Tq, H4, C3,
                  self.G(ln + '.weight_ih_l0'), C3, dbias=self.G(ln + '.bias_ih_l0') if fuse_b else None)
            wgrad(bwd, dgx_a.data_ptr(), Tq * H4, H4, _ptr(head['hseq'], (PAD_L - 1) * HP), head['gh'].Tp * HP, HP, B, Tq, H4,
                  HIDDEN, self.G(ln + '.weight_hh_l0'), HIDDEN, dbias=self.G(ln + '.bias_hh_l0') if fuse_b else None)
            # dX = dgx W_ih  (through the input dropout mask if any)
            if head['dmask'] is not None:
                epi = self._epi(C3, out2=gout.data_ptr(), mask2=head['dmask'], scale2=dscale, mask_rows=geo3.rows)
            else:
                epi = self._epi(C3, out=gout.data_ptr())
            gemm(bwd, dgx_a.data_ptr(), Tq * H4, H4, B, Tq, H4, C3, self.wt[ln].data_ptr(), H4, PAD_L, Tp3, 1, epi)
        else:
            dhp = zbuf(geo3.rows, C3, torch.float32)
            call(bwd, lib.nbasr_head_bwd, dt, _ptr(head['hsrc'], PAD_L * C3), Tp3 * C3, C3, B, Tq, C3, V, self.P(hn + '.weight'),
                 pl.dlogits.data_ptr(), _ptr(dhp, PAD_L * C3), Tp3 * C3, C3, self.G(hn + '.weight'), self.G(hn + '.bias'))
            epi = self._epi(C3, out=gout.data_ptr())
            call(bwd, lib.nbasr_eltwise, F32, dhp.data_ptr(), C3, B, Tq, Tp3, C3, C.byref(epi))
            pl.keep.append(epi)

        # Gradient buckets for the data-parallel exchange: (number of backward calls after which the flat-gradient range
        # [lo, hi) is final).  Parameters are laid out in module order (block 0 .. block 3, LSTM, classifier) and the backward
        # pass finishes them from the back, so each bucket is one contiguous range: head + LSTM first, then blocks 3..0.
        blk_lo = [self.slices[self.block_conv[i] + '.weight'][0] for i in range(4)]
        tail_lo = min(off for n_, (off, _) in self.slices.items() if off > blk_lo[3] and not n_.startswith(tuple(
            [self.block_conv[3] + '.', self.block_ln[3] + '.'] + [c + '.' for c in self.block_cells[3]])))
        pl.buckets = [(len(bwd), tail_lo, self.n_flat)]
        for i in (3, 2, 1, 0):
            rec = block_records[i]
            geo = rec['geo']
            Cc, Ti, Tp, mw = geo.C, geo.T, geo.Tp, geo.mw
            pool = pools[i]
            dz = dzs[i]
            for crec in reversed(rec['cells']):
                outs, nodes = crec['outs'], crec['nodes']
                nn_ = len(nodes)
                g = [None] * (nn_ + 1)
                dzb = [None] * nn_
                last = nodes[nn_ - 1]

                def need_g(mi):
                    # g[mi] (the gradient wrt outs[mi] itself) is read by the previous cell (mi = 0) or as the skip-connection
                    # contribution of node mi-1's branches; a branch-free conv / linear node only needs the GATED gradient dZ
                    return mi == 0 or any(nodes[mi - 1]['branches']) or nodes[mi - 1]['op'] == 'zero'

                # gradient wrt the pre-norm cell output o_n
                if m.use_norm:
                    g[nn_] = pool.pop()
                    dz_t = None
                    if last['op'] != 'zero':
                        dz_t = dz[nn_ - 1]
                        dzb[nn_ - 1] = dz_t
                    call(bwd, lib.nbasr_layernorm_bwd, dt, gout.data_ptr(), outs[nn_].data_ptr(), adt, S, crec['mean'].data_ptr(),
                         crec['rstd'].data_ptr(), self.P(crec['name'] + '.norm_layer.weight'), B, Ti, Tp, Cc,
                         g[nn_].data_ptr() if need_g(nn_) else None, dz_t.data_ptr() if dz_t is not None else None,
                         last['mask'].t.data_ptr() if dz_t is not None else None, dscale, geo.rows,
                         last['mask'].w if dz_t is not None else 32,
                         self.G(crec['name'] + '.norm_layer.weight'), self.G(crec['name'] + '.norm_layer.bias'))
                    pool.append(gout)
                else:
                    g[nn_] = gout
                    if last['op'] != 'zero':
                        dz_t = dz[nn_ - 1]
                        dzb[nn_ - 1] = dz_t
                        epi = self._epi(Cc, out2=dz_t.data_ptr(), mask2=last['mask'], scale2=dscale, mask_rows=geo.rows)
                        call(bwd, lib.nbasr_eltwise, dt, gout.data_ptr(), Cc, B, Ti, Tp, Cc, C.byref(epi))
                        pl.keep.append(epi)
                chain_wg = []

                def flush_bwd():
                    # weight gradients of the conv nodes since the last flush, after all of their input gradients
                    for a_ in chain_wg:
                        call(bwd, lib.nbasr_gconv_wgrad_x, *a_)
                    del chain_wg[:]

                for j in range(nn_ - 1, -1, -1):
                    nrec = nodes[j]
                    op, pn = nrec['op'], nrec['pn']
                    src = outs[j]
                    # contributions of later nodes' skip connections onto outs[j]
                    adds = [g[k + 1].data_ptr() for k in range(j, nn_) if nodes[k]['branches'][j]]
                    g[j] = pool.pop()
                    # the epilogue that produces g[j] also emits dZ_{j-1} = g[j] * mask_{j-1}
                    o2, m2 = 0, None
                    if j >= 1 and nodes[j - 1]['op'] != 'zero':
                        dzb[j - 1] = dz[j - 1]
                        o2, m2 = dzb[j - 1].data_ptr(), nodes[j - 1]['mask']
                    # (the un-gated gradient g[j] is written only when something reads it)
                    epi = self._epi(Cc, adds=adds, out=g[j].data_ptr() if (need_g(j) or not o2) else 0, out2=o2, mask2=m2, scale2=dscale,
                                    mask_rows=geo.rows)
                    if op not in CONV_EDGES:
                        flush_bwd()
                    if op == 'zero':
                        call(bwd, lib.nbasr_eltwise, dt, None, Cc, B, Ti, Tp, Cc, C.byref(epi))
                        pl.keep.append(epi)
                    elif op == 'linear':
                        d = dzb[j]
                        fuse = dt == BF16       # bias gradient rides on the tensor-core wgrad (ones operand)
                        wgrad(bwd, _ptr(d, PAD_L * Cc), Tp * Cc, Cc, _ptr(Bc(src), PAD_L * Cc), Tp * Cc, Cc, B, Ti, Cc, Cc,
                              self.G(pn + '.linear.weight'), Cc, dbias=self.G(pn + '.linear.bias') if fuse else None)
                        if not fuse:
                            call(bwd, lib.nbasr_colsum, dt, d.data_ptr(), B, Ti, Tp, Cc, self.G(pn + '.linear.bias'))
                        gemm(bwd, _ptr(d, PAD_L * Cc), Tp * Cc, Cc, B, Ti, Cc, Cc, self.wt[pn].data_ptr(), Cc, PAD_L, Tp, 1, epi)
                    else:
                        d = dzb[j]
                        k, dd, lp = nrec['k'], nrec['d'], nrec['lp']
                        # reads the forward activation itself: fp16 S*x in the 16-bit mode, un-scaled while it is staged
                        chain_wg.append((dt, d.data_ptr(), src.data_ptr(), adt, 1.0 / S, B, Ti, Tp, Cc, Cc // 100, k, -lp, dd,
                                         self.G(pn + '.conv.weight'), self.G(pn + '.conv.bias')))
                        gc = GConv()
                        gc.dtype, gc.x, gc.B, gc.T, gc.Tp, gc.C, gc.cpg = dt, d.data_ptr(), B, Ti, Tp, Cc, Cc // 100
                        gc.ktaps, gc.off0, gc.dstep, gc.w = k, lp - (k - 1) * dd, dd, self.wt[pn].data_ptr()
                        gc.w_packed = 3 if dt == BF16 else 0      # packed | stable
                        gc.epi = epi
                        call(bwd, lib.nbasr_gconv_fwd, C.byref(gc))
                        pl.keep.append(gc)
                flush_bwd()
                for k in range(1, nn_ + 1):   # (without norm, g[nn_] is the consumed incoming buffer)
                    pool.append(g[k])
                gout = g[0]
            # ---- top of the block: LayerNorm bwd -> dZ of the time-reduction conv
            dzc = dz[0]
            if i == 0:
                dz_blk0 = dzc
            lname, cname = self.block_ln[i], self.block_conv[i]
            call(bwd, lib.nbasr_layernorm_bwd, dt, gout.data_ptr(), rec['z'].data_ptr(), adt, S, rec['mean'].data_ptr(),
                 rec['rstd'].data_ptr(), self.P(lname + '.weight'), B, Ti, Tp, Cc, None, dzc.data_ptr(), rec['zmask'].t.data_ptr(),
                 1.0, geo.rows, 32, self.G(lname + '.weight'), self.G(lname + '.bias'))
            pool.append(gout)
            pgeo, s = rec['pg'], rec['s']
            fuse = dt == BF16
            wgrad(bwd, _ptr(dzc, PAD_L * Cc), Tp * Cc, Cc, rec['a_ptr'], pgeo.Tp * pgeo.C, s * pgeo.C, B, Ti, Cc, rec['K'],
                  self.G(cname + '.weight'), rec['K'], dbias=self.G(cname + '.bias') if fuse else None)
            if not fuse:
                call(bwd, lib.nbasr_colsum, dt, dzc.data_ptr(), B, Ti, Tp, Cc, self.G(cname + '.bias'))
            pl.buckets.append((len(bwd), blk_lo[i], blk_lo[i + 1] if i < 3 else tail_lo))
            if i > 0:
                gout = pools[i - 1].pop()
                Cin, Tin = pgeo.C, pgeo.T
                if s == 1:
                    epi = self._epi(Cin, out=gout.data_ptr())
                    gemm(bwd, _ptr(dzc, (PAD_L - 4) * Cc), Tp * Cc, Cc, B, Tin, 8 * Cc, Cin, self.wd[cname][0].data_ptr(), 8 * Cc,
                         PAD_L, pgeo.Tp, 1, epi)
                else:
                    for par in (0, 1):
                        nrp = (Tin - par + 1) // 2
                        epi = self._epi(Cin, out=gout.data_ptr())
                        gemm(bwd, _ptr(dzc, (PAD_L - 1 + par) * Cc), Tp * Cc, Cc, B, nrp, 4 * Cc, Cin,
                             self.wd[cname][par].data_ptr(), 4 * Cc, PAD_L + par, pgeo.Tp, 2, epi)
        pl.daudio = None
        if input_grad:
            # Gradient wrt the input features: block 0's stride-1 input-gradient GEMM (as for blocks > 0 above, C_in = 80),
            # fp32 output into a padded (B, Tp, 80) buffer, then back to the (B, 80, T) layout of the input.  The tap-flipped
            # operand of conv_0 belongs to this plan and is re-packed by it: the optimiser tail (and every CUDA graph
            # captured on it) keeps refreshing exactly the packs it refreshes without input gradients.
            rec = block_records[0]
            geo, cname = rec['geo'], self.block_conv[0]
            Cc, Tp = geo.C, geo.Tp
            wd0 = arena.zeros((FEATURES, 8 * Cc), tdt)
            call(bwd, lib.nbasr_pack_weight, self.P(cname + '.weight'), wd0.data_ptr(), dt, Cc, FEATURES, 8, 7, -1,
                 8 * FEATURES, 1, FEATURES)
            pl.dx_in = arena.zeros((g_in.rows, FEATURES), torch.float32)
            epi = self._epi(FEATURES, out=pl.dx_in.data_ptr(), out_dtype=F32)
            gemm(bwd, _ptr(dz_blk0, (PAD_L - 4) * Cc), Tp * Cc, Cc, B, T, 8 * Cc, FEATURES, wd0.data_ptr(), 8 * Cc, PAD_L,
                 g_in.Tp, 1, epi)
            pl.daudio = arena.zeros((B, FEATURES, T), torch.float32)
            call(bwd, lib.nbasr_transpose_out, pl.dx_in.data_ptr(), pl.daudio.data_ptr(), B, FEATURES, T, g_in.Tp)
            pl.in_geo = g_in
        pl.bwd = bwd
        return pl

    # ------------------------------------------------------------------ execution
    def _run(self, ops):
        st = torch.cuda.current_stream().cuda_stream
        for fn, args in ops:
            rc = fn(*args, st)
            if rc != 0:
                raise _lib.NbasrError(f'{fn.__name__}: {self.lib.nbasr_last_error().decode()}')
        # kernels launched: every C-ABI call launches >= 1 kernel of libnbasr
        self.launches += len(ops)

    @_on_device
    def forward(self, audio, training=None, grad=None, input_grad=False):
        """audio (B, 80, T) fp32 cuda -> plan (holds logits / logp buffers).  grad: a backward pass may follow;
        input_grad: it also computes pl.daudio, the gradient wrt `audio`."""
        self.bind()
        training = self.model.training if training is None else training
        B, F, T = audio.shape
        assert F == FEATURES
        pl = self.plan(B, T, training, grad, input_grad)
        self.refresh_packs()
        pl.audio.copy_(audio, non_blocking=True)
        if training and self.training_drop > 0:
            self.drop_step.add_(1)
        self._run(pl.fwd)
        return pl

    @_on_device
    def backward(self, pl, dlogits=None, zero_grad=True):
        if pl.bwd is None:
            raise RuntimeError('this plan was built for inference (grad=False): no gate masks / backward call list')
        if dlogits is not None:
            pl.dlogits.copy_(dlogits)
        if zero_grad:
            self.flat_g.zero_()
        self._run(pl.bwd)

    def attach_grads(self):
        """Re-point p.grad at the flat gradient buffer (torch's zero_grad(set_to_none=True) drops it)."""
        for name, p in zip(self.names, self.params):
            off, n = self.slices[name]
            if p.grad is None or p.grad.data_ptr() != self.flat_g.data_ptr() + 4 * off:
                gv = self.flat_g[off:off + n]
                if self._is_dense_conv_w(name):
                    co, ci, k = p.shape
                    p.grad = gv.view(co, k, ci).permute(0, 2, 1)
                else:
                    p.grad = gv.view(p.shape)

    @_on_device
    def set_lr(self, lr):
        if getattr(self, '_lr_host', None) != lr:   # device write only when the schedule changes lr
            self.opt_state[1:2].fill_(lr)
            self._lr_host = lr

    @_on_device
    def optimizer_step(self, lr, reg_coef=0.01, max_norm=5.0, betas=(0.9, 0.999), eps=1e-7):
        self.set_lr(lr)
        self._optimizer_launch(reg_coef, max_norm, betas, eps)

    def snapshot_state(self):
        return (self.flat_p.clone(), self.adam_m.clone(), self.adam_v.clone(), self.opt_state.clone(), self.drop_step.clone())

    @_on_device
    def restore_state(self, st):
        self.flat_p.copy_(st[0]); self.adam_m.copy_(st[1]); self.adam_v.copy_(st[2]); self.opt_state.copy_(st[3])
        self.drop_step.copy_(st[4])
        self.refresh_packs(force=True)

    def _optimizer_launch(self, reg_coef=0.01, max_norm=5.0, betas=(0.9, 0.999), eps=1e-7):
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(self.lib.nbasr_optim_step(self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.adam_m.data_ptr(),
                                             self.adam_v.data_ptr(), self.n_flat, self.seg_off.data_ptr(),
                                             self.seg_len.data_ptr(), int(self.seg_off.numel()), self.seg_chunks, reg_coef, max_norm,
                                             betas[0], betas[1], eps, self.opt_state.data_ptr(), st), 'optim')
        self.launches += 7 if self.seg_off.numel() else 4
        self.refresh_packs(force=True)


class ModelFunction(torch.autograd.Function):
    """Whole-model autograd node: forward/backward are engine plans, gradients land in the flat buffer."""

    @staticmethod
    def forward(ctx, model, audio, *params):
        eng = model.engine
        # gradients may be requested in eval mode too (dropout off): the plan then still records gate masks
        need = torch.is_grad_enabled() and (audio.requires_grad or any(p.requires_grad for p in eng.params))
        need_x = ctx.needs_input_grad[1]        # (grad mode is off inside Function.forward: ask autograd)
        pl = eng.forward(audio.contiguous().float(), grad=need or model.training, input_grad=need_x)
        ctx.eng, ctx.pl, ctx.audio_dtype = eng, pl, audio.dtype
        return pl.logits.clone()

    @staticmethod
    def backward(ctx, dlogits):
        eng, pl = ctx.eng, ctx.pl
        # Accumulate like autograd: the gradients of this call are added to whatever .grad holds.  A .grad can be (a) a
        # view of the flat gradient buffer (ours, from an earlier call) or (b) a fresh tensor another autograd node made
        # after optimizer.zero_grad(set_to_none=True) -- e.g. the conv-weight regulariser of the reference step
        # (trainer.py:221), whose norm nodes run before this one.  (b) is folded into the flat buffer, then re-pointed.
        views, foreign = False, []
        for name, p in zip(eng.names, eng.params):
            if p.grad is None:
                continue
            off, _ = eng.slices[name]
            if p.grad.data_ptr() == eng.flat_g.data_ptr() + 4 * off:
                views = True
            else:
                foreign.append((name, p, p.grad))
        saved = eng.flat_g.clone() if views else None
        eng.backward(pl, dlogits.contiguous(), zero_grad=True)
        if views:
            for name, p, _ in foreign:          # stale flat content under a foreign .grad is not a gradient of p
                off, n = eng.slices[name]
                saved[off:off + n].zero_()
            eng.flat_g.add_(saved)
        for name, p, g in foreign:
            off, n = eng.slices[name]
            dst = eng.flat_g[off:off + n]
            if eng._is_dense_conv_w(name):
                co, ci, k = p.shape
                dst.view(co, k, ci).add_(g.detach().to(dst.device, torch.float32).permute(0, 2, 1))
            else:
                dst.view(p.shape).add_(g.detach().to(dst.device, torch.float32))
        eng.attach_grads()
        # gradients were written in place into p.grad (views of the flat buffer); the input gradient is returned (autograd
        # accumulates it into audio.grad)
        daudio = pl.daudio.to(ctx.audio_dtype, copy=True) if pl.daudio is not None else None
        return (None, daudio) + tuple(None for _ in eng.params)
