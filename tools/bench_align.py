"""Time CTC forced alignment (nbasr_ctc_align) beside the CTC loss kernel (nbasr_ctc without and with dlogits) on one GPU.

    python tools/bench_align.py [--rounds 7] [--out profiles/align.json]

Shapes (output frames, blank = 0, V = 49, log-probs of random logits):
* cfg2_eval: 64 x 125, the eval step of bench.py's default workload (64 x 500 input frames, len_div 4), target lengths
  drawn as bench.py draws them (nb_asr_b200.data.make_batch, 20 <= S_b < 50);
* cfg5: 32 x 750 (32 x 3 000 input frames, every row at full length), 150 <= S_b <= 300 (up to L = 601 states; the
  backpointers still fit in shared memory).
Each kernel's launches are captured in one CUDA graph (so the host's per-call cost does not hide the kernel), the graph
replay is timed with CUDA events, the three kernels alternate for `--rounds` rounds, and the median, min and max per
launch are reported.  The inputs (1.6 MB / 4.7 MB of log-probs) stay resident in the 126 MB L2 between launches, as they
are when these kernels follow the classifier in an eval step.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nb_asr_b200 import _lib, data  # noqa: E402

V = 49
SHAPES = {'cfg2_eval': dict(B=64, frames=500, min_len=500, tgt_lo=20, tgt_hi=50, launches=400),
          'cfg5': dict(B=32, frames=3000, min_len=3000, tgt_lo=150, tgt_hi=301, launches=100)}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def kernels(shape, dev):
    """(name -> zero-argument launcher) on one batch of the shape; every launcher enqueues exactly one library call."""
    lib = _lib.load()
    (_, alen), (tg, tl) = data.make_batch(shape['B'], shape['frames'], seed=0, min_len=shape['min_len'],
                                          tgt_lo=shape['tgt_lo'], tgt_hi=shape['tgt_hi'])
    B, S, T = tg.shape[0], tg.shape[1], shape['frames'] // 4
    g = torch.Generator(device=dev).manual_seed(0)
    logp = torch.log_softmax(3.0 * torch.randn(B, T, V, generator=g, device=dev), -1).contiguous()
    alen, tg, tl = alen.to(dev), tg.to(dev).contiguous(), tl.to(dev)
    L = 2 * S + 1
    work = torch.empty(2 * B * T * L + 16, device=dev)
    nll, loss, dl = torch.empty(B, device=dev), torch.empty(1, device=dev), torch.empty(B, T, V, device=dev)
    i32 = dict(dtype=torch.int32, device=dev)
    out = [torch.empty(B, T, **i32), torch.empty(B, T, **i32), torch.empty(B, S, **i32), torch.empty(B, S, **i32),
           torch.empty(B, device=dev)]
    nwork = lib.nbasr_ctc_align_work_bytes(B, T, S)
    awork = torch.empty(max(1, nwork), dtype=torch.uint8, device=dev)
    p = lambda t: t.data_ptr()  # noqa: E731
    st = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731

    def ctc(dlogits):
        return lambda: _lib.check(lib.nbasr_ctc(p(logp), B, T, V, p(tg), S, p(alen), 4, p(tl), p(nll), p(loss),
                                                p(dl) if dlogits else None, p(work), st()), 'ctc')

    def align():
        _lib.check(lib.nbasr_ctc_align(p(logp), B, T, V, p(tg), S, p(alen), 4, p(tl), *map(p, out), p(awork), st()),
                   'ctc_align')

    meta = dict(B=B, T=T, V=V, S=S, S_b_range=[int(tl.min()), int(tl.max())], backpointers='work' if nwork else 'shared memory')
    return {'ctc_align': align, 'ctc': ctc(False), 'ctc+dlogits': ctc(True)}, meta


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_align needs a GPU')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    res = {'gpu': gpu_info(), 'method': 'CUDA events around the replay of a graph of back-to-back launches, kernels alternated '
           'per round', 'shapes': {}}
    for name, shape in SHAPES.items():
        fns, meta = kernels(shape, dev)
        n = shape['launches']
        graphs = {}
        for k, f in fns.items():
            for _ in range(10):          # warm-up: module load, function attributes
                f()
            torch.cuda.synchronize()
            graphs[k] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphs[k]):
                for _ in range(n):
                    f()
            graphs[k].replay()
        torch.cuda.synchronize()
        per = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, g in graphs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize()
                per[k].append(e0.elapsed_time(e1) * 1e3 / n)
        meta['launches_per_round'] = n
        meta['us_per_launch'] = {k: {'median': round(statistics.median(v), 2), 'min': round(min(v), 2), 'max': round(max(v), 2)}
                                 for k, v in per.items()}
        res['shapes'][name] = meta
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
