"""Per-launch timing of an engine plan with CUDA events (on the launching stream) + algorithmic work model.

Used by bench.py for the live roofline figure and by tools/ for optimisation work.  Algorithmic
FLOPs / bytes follow SURVEY.md §8(d) / DESIGN.md "Kernels and rooflines".
"""
import collections
import ctypes as C

import torch

from . import _lib
from ._lib import BF16, GConv, Gemm, Wgrad


def _struct_of(arg, typ):
    # ctypes.byref objects keep the referenced struct in ._obj
    obj = getattr(arg, '_obj', None)
    return obj if isinstance(obj, typ) else None


def op_work(fn_name, args, es):
    """(class tag, algorithmic flops, algorithmic bytes) of one plan entry. es = activation element size."""
    if fn_name == 'nbasr_gemm_tn':
        g = _struct_of(args[0], Gemm)
        rows = g.nb * g.nr
        flops = 2.0 * rows * g.K * g.N
        a_cols = min(g.K, g.a_rs) if g.a_rs > 0 else g.K      # overlapping rows are read once
        # (an out2 without a gate mask is the bf16 twin of `out` for the weight gradient: an implementation cost of the
        # fp16-forward / bf16-backward split, not algorithmic traffic)
        n_o = g.epi.n_add + (1 if g.epi.out else 0) + (1 if (g.epi.out2 and g.epi.mask2) else 0)
        byts = rows * a_cols * es + g.N * g.K * es + rows * g.N * es * n_o
        return f'gemm_tn K={g.K} N={g.N}', flops, byts
    if fn_name == 'nbasr_gemm_wgrad':
        w = _struct_of(args[0], Wgrad)
        rows = w.nb * w.nr
        flops = 2.0 * rows * w.M * w.N
        x_cols = min(w.N, w.x_rs)
        byts = rows * (w.M + x_cols) * es + 4.0 * w.M * w.N * 2
        return f'gemm_wgrad M={w.M} N={w.N}', flops, byts
    if fn_name == 'nbasr_gconv_fwd':
        g = _struct_of(args[0], GConv)
        el = g.B * g.T * g.C
        n_t = 1 + g.epi.n_add + (1 if g.epi.out else 0) + (1 if (g.epi.out2 and g.epi.mask2) else 0)     # tensors read/written once
        n_m = (1 if g.epi.mask_out else 0) + (1 if g.epi.mask2 else 0)                 # 1 bit / element each
        return f'gconv C={g.C} k={g.ktaps} d={g.dstep}', 2.0 * el * g.cpg * g.ktaps, el * es * n_t + el * n_m / 8.0
    if fn_name == 'nbasr_gconv_chain':
        # a chain launch processes n nodes: algorithmic work = the sum of its nodes' (SURVEY.md 8d per-node figures)
        fl = by = 0.0
        for i in range(args[1]):
            _, f1, b1 = op_work('nbasr_gconv_fwd', (C.byref(args[0][i]),), es)
            fl, by = fl + f1, by + b1
        g = args[0][0]
        return f'gconv C={g.C} chain of {args[1]}', fl, by
    if fn_name in ('nbasr_gconv_wgrad', 'nbasr_gconv_wgrad_x'):
        B, T, Tp, Cc, cpg, k = args[3:9] if fn_name == 'nbasr_gconv_wgrad' else args[5:11]
        el = B * T * Cc
        return f'gconv_wgrad C={Cc} k={k}', 2.0 * el * cpg * k, el * es * 2
    if fn_name in ('nbasr_layernorm_fwd', 'nbasr_layernorm_bwd'):
        if fn_name.endswith('fwd'):
            B, T, Tp, Cc = args[3:7]
            return f'ln_fwd C={Cc}', 0.0, B * T * Cc * es * 2
        B, T, Tp, Cc = args[8:12]
        n_out = (1 if args[12] else 0) + (1 if args[13] else 0)
        return f'ln_bwd C={Cc}', 0.0, B * T * Cc * es * (2 + n_out)
    if fn_name == 'nbasr_eltwise':
        B, T, Tp, Cc = args[3:7]
        return f'eltwise C={Cc}', 0.0, B * T * Cc * es * 2
    if fn_name == 'nbasr_colsum':
        B, T, Tp, Cc = args[2:6]
        return f'colsum C={Cc}', 0.0, B * T * Cc * (2 if args[0] == BF16 else 4)
    return fn_name.replace('nbasr_', ''), 0.0, 0.0


def gconv_issue_floor_cycles(fn_name, args):
    """Structural floor of the tcgen05 grouped-conv forward / input-gradient kernel (DESIGN.md 3.1): 3*k MMAs of N = 48 per
    128-frame x 48-channel tile, each >= 88 cycles of tensor-pipe issue (both operands in shared memory), on one SM."""
    if fn_name == 'nbasr_gconv_chain':
        return sum(gconv_issue_floor_cycles('nbasr_gconv_fwd', (C.byref(args[0][i]),)) for i in range(args[1]))
    if fn_name != 'nbasr_gconv_fwd':
        return 0.0
    g = _struct_of(args[0], GConv)
    out = 40 if g.cpg == 10 else 48
    tiles = -(-g.C // out) * g.B * -(-g.T // 128)
    return tiles * 3.0 * g.ktaps * 88.0


def profile_ops(engine, ops, iters=3):
    """Time every entry of a plan op list. Returns {tag: dict(n, ms, flops, bytes)} averaged over iters."""
    st = torch.cuda.current_stream()
    es = 2 if engine.dt == BF16 else 4          # 16-bit mode: fp16 activations and bf16 gradients are both 2 bytes
    n = len(ops)
    acc = collections.OrderedDict()
    for it in range(iters + 1):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        evs[0].record(st)
        for i, (fn, args) in enumerate(ops):
            _lib.check(fn(*args, st.cuda_stream), fn.__name__)
            evs[i + 1].record(st)
        torch.cuda.synchronize()
        if it == 0:
            continue   # warm-up pass
        for i, (fn, args) in enumerate(ops):
            tag, fl, by = op_work(fn.__name__, args, es)
            d = acc.setdefault(tag, dict(n=0, ms=0.0, flops=0.0, bytes=0.0, floor_cycles=0.0))
            d['floor_cycles'] += gconv_issue_floor_cycles(fn.__name__, args)
            # kernel launches of this entry (an unfused grouped-conv chain launches one kernel per node)
            d['n'] += args[1] if (fn.__name__ == 'nbasr_gconv_chain' and not args[2]) else 1
            d['ms'] += evs[i].elapsed_time(evs[i + 1])
            d['flops'] += fl
            d['bytes'] += by
    for d in acc.values():
        for k in d:
            d[k] /= iters
    return acc


def format_profile(acc, top=40):
    tot = sum(d['ms'] for d in acc.values())
    lines = [f'{"class":38s} {"n":>4s} {"ms":>8s} {"%":>6s} {"TFLOP/s":>8s} {"GB/s":>8s}']
    for tag, d in sorted(acc.items(), key=lambda kv: -kv[1]['ms'])[:top]:
        tf = d['flops'] / d['ms'] / 1e9 if d['ms'] > 0 else 0
        gb = d['bytes'] / d['ms'] / 1e6 if d['ms'] > 0 else 0
        lines.append(f'{tag:38s} {d["n"]:4.0f} {d["ms"]:8.3f} {100 * d["ms"] / tot:6.1f} {tf:8.1f} {gb:8.0f}')
    lines.append(f'{"total":38s} {"":4s} {tot:8.3f}')
    return '\n'.join(lines)
