"""Time the zero-cost proxies (nb_asr_b200.proxies) on one GPU.

    python tools/bench_proxies.py [--reps 5] [--sample 24] [--out profiles/proxies.json]

* ms per measure (grad_norm and snip share one forward + backward and are timed together) for four archs at B x T = 64 x 500;
  nwot alone (one forward pass + nbasr_gate_gram) and grad_norm + snip + nwot (nwot reuses their forward pass); zico
  alone (two half-batch forward + backward passes + nbasr_grad_snr);
* nbasr_grad_snr alone (CUDA events) on each arch's own two gradient snapshots (N = 2) and the bytes it reads;
* the sweep's candidates per second on a fixed sample of unique archs (every k-th of the 8 242), evaluated exactly as
  nb_asr_b200.sweep does, without proxies, with --proxies nwot, with all five proxies and with --proxies zico
  (--proxy-batches 1), and the Kendall tau between the zico columns of the 16-bit and the fp32 sweep;
* the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nb_asr_b200 as nb  # noqa: E402
from nb_asr_b200 import _lib, data, graph_utils, proxies, sweep  # noqa: E402

ARCHS = {'default': [[1, 0], [1, 0, 0], [1, 0, 0, 0]], 'linear_skips': [[0, 1], [0, 1, 1], [0, 1, 1, 1]],
         'c7d2_skips': [[4, 1], [4, 1, 1], [4, 1, 1, 1]], 'zero_mix': [[5, 1], [1, 1, 0], [5, 0, 1, 1]]}
GROUPS = {'grad_norm+snip': ('grad_norm', 'snip'), 'jacob_cov': ('jacob_cov',), 'synflow': ('synflow',), 'nwot': ('nwot',),
          'grad_norm+snip+nwot': ('grad_norm', 'snip', 'nwot'), 'zico': ('zico',)}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def time_measures(arch, precision, reps, B=64, T=500):
    model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=0, precision=precision, init='device', seed=1235,
                         conv_gain=101 ** 0.5).eval()
    b = data.make_batch(B, T, seed=0, min_len=T // 2)
    b = ((b[0][0].cuda(), b[0][1].cuda()), (b[1][0].cuda(), b[1][1].cuda()))
    res = {}
    for g, ms in GROUPS.items():
        for _ in range(2):
            vals = proxies.compute_proxies(model, b, ms)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            proxies.compute_proxies(model, b, ms)
        torch.cuda.synchronize()
        res[g] = (time.perf_counter() - t0) / reps * 1e3
        res.update({f'value_{k}': v for k, v in vals.items()})
    # nbasr_gate_gram alone, on the masks of the forward pass nwot just ran (CUDA events)
    eng = model.engine
    pl = eng.plan(B, T, False, True)
    alen = b[0][1].to(torch.int64).contiguous()
    proxies._gate_gram(eng, pl, alen)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        proxies._gate_gram(eng, pl, alen)
    e1.record()
    torch.cuda.synchronize()
    res['gate_gram_call'] = e0.elapsed_time(e1) / reps
    res['relu_layers'] = len(pl.gates)
    # nbasr_grad_snr alone on the model's own N = 2 snapshots (CUDA events)
    snaps = proxies.zico_snapshots(model, b, 2)
    names = proxies.scored_names(model)
    off, ln, chunks, part, out = proxies._segments(eng, names)
    st = torch.cuda.current_stream().cuda_stream

    def snr():
        _lib.check(eng.lib.nbasr_grad_snr(snaps.data_ptr(), snaps.stride(0), 2, off.data_ptr(), ln.data_ptr(), len(names),
                                          chunks, part.data_ptr(), out.data_ptr(), st), 'grad_snr')
    snr()
    e0.record()
    for _ in range(20 * reps):
        snr()
    e1.record()
    torch.cuda.synchronize()
    res['grad_snr_us'] = e0.elapsed_time(e1) / (20 * reps) * 1e3
    res['grad_snr_params'] = int(ln.sum())
    res['grad_snr_GB_per_s'] = 2 * 4 * res['grad_snr_params'] / (res['grad_snr_us'] * 1e3)
    model._engine = None
    return res


def sweep_rate(archs, batches, measures, precision='bf16'):
    kw = dict(proxies=measures, proxy_batches=1) if measures else {}
    n_ref = sum(int(tl.sum()) for _, (t, tl) in batches)
    sweep.evaluate_arch(archs[0], batches, 0, precision, init='device', conv_gain=101 ** 0.5, n_ref=n_ref, **kw)   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rows = [sweep.evaluate_arch(a, batches, 0, precision, init='device', conv_gain=101 ** 0.5, n_ref=n_ref, **kw) for a in archs]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return len(archs) / dt, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--sample', type=int, default=24)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = dict(gpu=gpu_info(), B=64, T=500, measures_ms={})
    for name, arch in ARCHS.items():
        for precision in ('bf16', 'fp32'):
            r = time_measures(arch, precision, args.reps)
            out['measures_ms'][f'{name}/{precision}'] = r
            print(json.dumps({f'{name}/{precision}': r}), flush=True)
    uniq = [a for _, a in graph_utils.get_unique_architectures()]
    step = max(1, len(uniq) // args.sample)
    archs = uniq[::step][:args.sample]
    batches = data.timit_shaped_eval_set(n_utt=1344, batch_size=64, seed=0)
    batches = [((a.cuda(), al.cuda()), (t.cuda(), tl.cuda())) for (a, al), (t, tl) in batches]
    r0, _ = sweep_rate(archs, batches, ())
    rn, _ = sweep_rate(archs, batches, ('nwot',))
    r1, rows = sweep_rate(archs, batches, proxies.MEASURES)
    finite = {m: sum(r[m] == r[m] and abs(r[m]) != float('inf') for r in rows) for m in proxies.MEASURES}
    rz, rows_z = sweep_rate(archs, batches, ('zico',))
    rz32, rows_z32 = sweep_rate(archs, batches, ('zico',), precision='fp32')
    z16, z32 = [r['zico'] for r in rows_z], [r['zico'] for r in rows_z32]
    from scipy.stats import kendalltau
    out['sweep'] = dict(n_archs=len(archs), sample_step=step, archs_per_s=r0, archs_per_s_with_nwot=rn,
                        archs_per_s_with_proxies=r1, measures=list(proxies.MEASURES), rows_with_finite=finite,
                        archs_per_s_with_zico=rz, archs_per_s_with_zico_fp32=rz32,
                        zico_kendall_tau_bf16_vs_fp32=float(kendalltau(z16, z32)[0]), zico_bf16=z16, zico_fp32=z32,
                        eval_batches=len(batches), proxy_batches=1)
    print(json.dumps(out['sweep']), flush=True)
    print(json.dumps(dict(gpu=out['gpu'])))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, 'w'), indent=1)


if __name__ == '__main__':
    main()
