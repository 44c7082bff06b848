#!/usr/bin/env python
"""Headline benchmark: NAS-Bench-ASR candidate TRAIN step (fwd + CTC + bwd + reg + clip + Adam) throughput.

    python bench.py --gpus N --steps K --warmup W            # ours (one process per GPU under torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own torch code on the host CPU cores

Workload of `value` (BASELINE.json configs[1]): arch [[1,0],[1,0,0],[1,0,0,0]], batch 64 x 500 frames x 80 log-mel per
GPU, 16-bit tensor-core operands with fp32 accumulation, fp32 LayerNorm statistics / LSTM state / CTC.  Synthetic
N(0,1) log-mel, U{1..48} labels, weights from seed 1235 (SURVEY.md §8d).  Prints ONE JSON line on rank 0.  Besides the
contract keys the line carries `cfg1` (configs[0]: B=8 eval + greedy PER, GPU beside the reference on the CPU) and
`cfg3` (configs[2]: the conv7d2+skips and the all-linear archs, data-parallel at this N).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_ARCH = [[1, 0], [1, 0, 0], [1, 0, 0, 0]]
ARCHS = {'default': DEFAULT_ARCH, 'c7d2_skips': [[4, 1], [4, 1, 1], [4, 1, 1, 1]],
         'linear_skips': [[0, 1], [0, 1, 1], [0, 1, 1, 1]], 'mixed': [[2, 1], [3, 0, 1], [0, 1, 0, 1]]}
REF_BUDGET_S = 200.0        # the reference arm sizes its per-step sample so that (W + K) steps fit this budget


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--arch', default='default')
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--frames', type=int, default=500)
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--dropout', type=float, default=0.0)
    ap.add_argument('--profile', action='store_true', help='print the per-kernel-class breakdown to stderr')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the cfg1 / cfg3 side measurements')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the loss, log-probs and output lengths of the last timed train step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy in float32 / float64.  An array larger than its share of DUMP_LIMIT_BYTES is
    replaced by a fixed sample of its elements (same positions for the same shape), so two builds compare element for
    element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.itemsize * a.size > share:
            idx = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, f'{name}.npy'), a)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sust=d['bf16_tflops_sustained'], src='measured')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        time.sleep(0.05)
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------ reference (CPU)
class CpuReference:
    """The reference's own torch implementation of the step on the host cores.  kind = "reference": the UNMODIFIED
    package installed into baseline/_ref (oracle/install_reference.sh) behind the four import shims of
    oracle/reference_shims.py; kind = "port": oracle/model_ref.py (the restatement pinned to it by tests/golden) when the
    installed copy is absent.  Greedy decode + fold + PER is the numpy restatement in both cases (the reference's decode
    lives in the third-party ctcdecode / torch_edit_distance packages, which are not installed)."""

    def __init__(self, arch):
        import torch
        from oracle import model_ref as M
        self.torch, self.M, self.arch = torch, M, arch
        torch.set_num_threads(os.cpu_count() or 1)
        self.cores = os.cpu_count() or 1
        self.kind = 'port'
        try:
            from oracle import reference_shims as R
            if R.find_reference():
                self.nb = R.import_reference()
                self.nb.set_seed(1235)
                self.model = self.nb.get_model(arch, use_rnn=True, dropout_rate=0.0)
                self.tr = R.reference_trainer(self.nb, self.model)
                self.kind = 'reference'
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f'[bench] installed reference unusable ({e!r}); timing the oracle port instead\n')
        if self.kind == 'port':
            self.sd = M.build_state_dict(arch, seed=1235)
            self.opt = None

    def batch(self, B, T):
        return self.M.make_batch(B, T, seed=0, min_len=T, tgt_lo=20, tgt_hi=50)

    def train_step(self, batch):
        audio, alen, tg, tl = batch
        t0 = time.perf_counter()
        if self.kind == 'reference':
            self.model.train()
            loss, _, _ = self.tr.step(((audio, alen), (tg, tl)), training=True)
        else:
            loss, _, _, _, self.sd, self.opt, _ = self.M.train_step(self.sd, self.arch, audio, alen, tg, tl, self.opt)
        float(loss)
        return time.perf_counter() - t0

    def eval_step(self, batch):
        """cfg 1: forward + log_softmax + CTC loss (reference Trainer.step(training=False)) + greedy decode + fold + PER."""
        from oracle import decode_np as D
        audio, alen, tg, tl = batch
        t0 = time.perf_counter()
        with self.torch.no_grad():
            if self.kind == 'reference':
                self.model.eval()
                loss, logp, out_len = self.tr.step(((audio, alen), (tg, tl)), training=False)
            else:
                loss, logp, out_len, _ = self.M.eval_step(self.sd, self.arch, audio, alen, tg, tl)
        per, dist, _, _ = D.per_batch(logp.numpy(), out_len.numpy(), tg.numpy(), tl.numpy())
        return time.perf_counter() - t0, float(loss), float(per), dist


def run_reference(args, arch, rank):
    """--impl reference: each step = one full train step of the reference on a bounded sample of the workload (the whole
    batch when (W + K) steps of it fit REF_BUDGET_S on this host, else the largest of 32 / 16 / 8 utterances that does)."""
    if rank != 0:
        return
    ref = CpuReference(arch)
    t8 = ref.train_step(ref.batch(8, args.frames))            # probe (also warms the thread pool / allocator)
    t8 = min(t8, ref.train_step(ref.batch(8, args.frames)))
    n_steps = max(1, args.steps) + max(0, args.warmup)
    Bs = 8
    for cand in (args.batch, 32, 16):
        if cand <= args.batch and 1.25 * t8 * cand / 8 * n_steps <= REF_BUDGET_S:
            Bs = cand
            break
    batch = ref.batch(Bs, args.frames)
    times = []
    for i in range(n_steps):
        t = ref.train_step(batch)
        if i >= args.warmup:
            times.append(t)
    t = sum(times) / len(times)
    val = Bs / t
    sample = (f'each step = one full train step (fwd+CTC+bwd+reg+clip+Adam) of the {"unmodified reference (baseline/_ref)" if ref.kind == "reference" else "oracle port"} '
              f'on {Bs} of the {args.batch} utterances ({Bs}x{args.frames}x80), fp32, {ref.cores} host threads')
    cfg = workload_config(args, arch, 1)
    cfg['reference_sample_batch'] = Bs
    print(json.dumps({
        'impl': 'reference', 'metric': 'train_utterances_per_sec', 'value': val, 'unit': 'utt/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
        'cpu_baseline': {'value': val, 'unit': 'utt/s', 'cores': ref.cores, 'kind': ref.kind, 'sample': sample},
        'e2e': {'value': val, 'unit': 'utt/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


def workload_config(args, arch, world):
    return {'workload': f'train step (fwd+CTC+bwd+reg+clip+Adam), arch {arch}, batch {args.batch}x{args.frames} frames x80 log-mel per GPU',
            'arch_vec': arch, 'per_gpu_batch': args.batch, 'global_batch': args.batch * world, 'frames': args.frames,
            'parallelism': f'dp{world} (utterance-sharded; the flat fp32 gradient is all-reduced by NCCL in 5 buckets overlapped with the backward pass)' if world > 1 else 'single GPU',
            'l2': 'per-step working set (activations + weights) is > 2 GB, far above the 126 MB L2; no flush needed',
            'dropout': args.dropout}


# ------------------------------------------------------------------------------------------------ ours (GPU)
def main():
    args = parse()
    arch = ARCHS.get(args.arch) or json.loads(args.arch)
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, arch, rank)
        return
    import torch
    import torch.distributed as dist
    import nb_asr_b200 as nb
    from nb_asr_b200 import profiling
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # NCCL_DEBUG / NCCL_DEBUG_FILE are left exactly as the caller set them (the driver reads the rank count there)
        dist.init_process_group('nccl', device_id=dev)
    B, T = args.batch, args.frames

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, eng=None):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = eng.launches if eng is not None else 0
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        timed.launches = (eng.launches - n0) if eng is not None else 0
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def build(arch_, precision, batch, frames, seed_off=0):
        nb.set_seed(1235)
        model = nb.get_model(arch_, use_rnn=True, dropout_rate=args.dropout, gpu=local, precision=precision)
        model.train()
        tr = nb.get_trainer((nb.PhonemeEncoder(48), None, None, None), nb.get_loss(), gpus=[local], verbose=False)
        tr.model = tr._model = model
        tr.optimizer = nb.trainer.FusedAdam(model, lr=1e-4)
        tr.use_graph = not args.no_graph
        (audio, alen), (tg, tl) = nb.data.make_batch(batch, frames, seed=rank + seed_off, min_len=frames, tgt_lo=20, tgt_hi=50, pin=True)
        host = ((audio, alen), (tg, tl))
        devb = ((audio.to(dev), alen.to(dev)), (tg.to(dev), tl.to(dev)))
        return model, tr, host, devb

    model, tr, host_batch, dev_batch = build(arch, args.precision, B, T)
    (audio, alen), (tg, tl) = host_batch
    eng = model.engine

    # ---- device-resident throughput (value)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last = {}

    def train_step():
        last['out'] = tr.step(dev_batch, training=True)
    ms = timed(train_step, args.steps, max(3, args.warmup), eng)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        loss, logp, out_len = last['out']
        dump_outputs(args.dump_outputs, {'loss': loss.double().cpu().numpy(), 'log_probs': logp.float().cpu().numpy(),
                                         'out_len': out_len.double().cpu().numpy()})
    launches_total = timed.launches
    ms_step = ms / args.steps
    value = world * B * args.steps / (ms / 1e3)

    # ---- end to end: pinned host inputs -> step -> loss on host, every step
    def e2e_step():
        loss, _, _ = tr.step(host_batch, training=True)
        return loss.item()
    ms_e2e = timed(e2e_step, args.steps, 3, eng)
    e2e_val = world * B * args.steps / (ms_e2e / 1e3)
    h2d = sum(t.numel() * t.element_size() for t in (audio, alen, tg, tl))

    # ---- eval step (fwd + CTC loss + greedy decode + PER), audio-seconds per second
    model.eval()

    def eval_step():
        loss, logp, out_len = tr.step(dev_batch, training=False)
        return tr.decode(logp, out_len, dev_batch)
    ms_eval = timed(eval_step, args.steps, 3, eng)
    audio_s = float(alen.sum()) / 100.0
    eval_val = world * audio_s * args.steps / (ms_eval / 1e3)
    model.train()

    # ---- live per-kernel timing (CUDA events on the launching stream) for the roofline entry (rank 0)
    roofline = None
    if rank == 0:
        roofline = roofline_entry(args, torch, profiling, eng, B, T, clocks, dev)
    barrier()
    del model, tr, eng
    torch.cuda.empty_cache()

    # ---- cfg 3 (BASELINE.json configs[2]): the named largest-FLOP arch (all conv7d2 + all skips) and the true one
    #      (all linear + all skips, SURVEY finding 1), same per-GPU batch, data-parallel at this N
    cfg3 = None
    if not args.no_extra and args.arch == 'default':
        cfg3 = {}
        for name in ('c7d2_skips', 'linear_skips'):
            m3, t3, _, db3 = build(ARCHS[name], args.precision, B, T)
            n3 = args.steps
            ms3 = timed(lambda: t3.step(db3, training=True), n3, 3, m3.engine)
            cfg3[name] = {'arch_vec': ARCHS[name], 'ms_per_step': ms3 / n3, 'value': world * B * n3 / (ms3 / 1e3), 'unit': 'utt/s',
                          'grad_bytes_per_step': 4 * int(m3.engine.n_flat), 'gpu_launches_per_step': timed.launches / n3}
            del m3, t3, db3
            torch.cuda.empty_cache()

    # ---- cfg 1 (BASELINE.json configs[0]): B=8 x 500 eval step + greedy PER, GPU (both precisions) beside the reference
    cfg1 = None
    if not args.no_extra and args.arch == 'default' and rank == 0 and world == 1:
        cfg1 = cfg1_entry(args, torch, nb, build, timed, dev)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(arch)
        Bc = 8
        cb = ref.batch(Bc, T)
        ref.train_step(cb)
        ts = [ref.train_step(cb) for _ in range(3)]
        t = sum(ts) / len(ts)
        cpu = {'value': Bc / t, 'unit': 'utt/s', 'cores': ref.cores, 'kind': ref.kind,
               'sample': f'3 timed train steps (after 1 warm-up) on {Bc} of the {B} utterances ({Bc}x{T}x80), fp32, '
                         f'{"unmodified reference package (baseline/_ref) through its own Trainer.step" if ref.kind == "reference" else "oracle port of the reference step"}, '
                         f'all host threads'}

    out = {'metric': 'train_utterances_per_sec', 'value': value, 'unit': 'utt/s', 'n_gpus': world, 'steps': args.steps,
           'warmup': max(3, args.warmup), 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': 'bf16' if args.precision == 'bf16' else 'f32', 'data': 'synthetic',
           'config': workload_config(args, arch, world), 'clocks': clocks,
           'e2e': {'value': e2e_val, 'unit': 'utt/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4, 'ms_per_step': ms_e2e / args.steps},
           'gpu_launches': launches_total,
           'eval': {'metric': 'eval_audio_seconds_per_sec', 'value': eval_val, 'unit': 'audio-s/s', 'ms_per_step': ms_eval / args.steps},
           'roofline': roofline, 'cpu_baseline': cpu, 'cfg1': cfg1, 'cfg3': cfg3}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def cfg1_entry(args, torch, nb, build, timed, dev):
    """configs[0]: arch default, fwd + CTC loss + greedy PER, batch 8 x 500 x 80.  GPU eval audio-s/s in both precisions,
    the reference on the host cores, and the parity facts of this exact config (loss, PER, edit distances)."""
    B1, T1 = 8, 500
    out = {'workload': f'arch {DEFAULT_ARCH} eval step: fwd + log_softmax + CTC loss + greedy decode + fold + PER, batch {B1}x{T1}x80'}
    res = {}
    for prec in ('fp32', 'bf16'):
        m1, t1, hb, db = build(DEFAULT_ARCH, prec, B1, T1, seed_off=0)
        m1.eval()
        state = {}

        def ev():
            loss, logp, ol = t1.step(db, training=False)
            state['loss'] = loss
            return t1.decode(logp, ol, db)
        n1 = args.steps
        ms1 = timed(ev, n1, 3, m1.engine)
        per = ev()
        audio_s = float(hb[0][1].sum()) / 100.0
        res[prec] = dict(loss=float(state['loss'].item()), per=float(per.item()), dist=t1.last_hyp[2].cpu().tolist())
        out[f'gpu_{prec}'] = {'value': audio_s * n1 / (ms1 / 1e3), 'unit': 'audio-s/s', 'ms_per_step': ms1 / n1,
                              'utt_per_s': B1 * n1 / (ms1 / 1e3)}
        del m1, t1
        torch.cuda.empty_cache()
    if not args.no_cpu_baseline:
        ref = CpuReference(DEFAULT_ARCH)
        audio, alen, tg, tl = ref.batch(B1, T1)         # same generator as nb.data.make_batch(seed=0): identical batch
        cb = (audio, alen, tg, tl)
        ref.eval_step(cb)
        rs = [ref.eval_step(cb) for _ in range(5)]
        t = sorted(r[0] for r in rs)[len(rs) // 2]
        _, rloss, rper, rdist = rs[-1]
        out['cpu'] = {'value': float(alen.sum()) / 100.0 / t, 'unit': 'audio-s/s', 'ms_per_step': 1e3 * t, 'utt_per_s': B1 / t,
                      'cores': ref.cores, 'kind': ref.kind, 'sample': '1 warm-up + median of 5 eval steps on the whole 8x500x80 batch'}
        out['parity'] = {'loss_reference': rloss, 'loss_gpu_fp32': res['fp32']['loss'], 'loss_gpu_16bit': res['bf16']['loss'],
                         'per_reference': rper, 'per_gpu_fp32': res['fp32']['per'], 'per_gpu_16bit': res['bf16']['per'],
                         'edit_distances_equal_fp32': res['fp32']['dist'] == [int(x) for x in rdist],
                         'edit_distances_equal_16bit': res['bf16']['dist'] == [int(x) for x in rdist]}
    return out


def roofline_entry(args, torch, profiling, eng, B, T, clocks, dev):
    pl = eng.plan(B, T, True)
    prof = profiling.profile_ops(eng, pl.fwd + pl.bwd, iters=3)
    # optimiser tail (regulariser + clip + Adam + operand re-pack), timed as one unit on the launching stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    eng._optimizer_launch()
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(3):
        eng._optimizer_launch()
    ev[1].record()
    torch.cuda.synchronize()
    n_par = float(eng.n_flat)
    prof['optim+repack'] = dict(ms=ev[0].elapsed_time(ev[1]) / 3, flops=0.0, bytes=n_par * (4 * 7 + 2 * 2), n=1.0)
    if args.profile:
        sys.stderr.write(profiling.format_profile(prof) + '\n')
    fam = {}
    for tag, d in prof.items():
        f = fam.setdefault(tag.split(' ')[0], dict(ms=0.0, flops=0.0, bytes=0.0, n=0, floor_cycles=0.0))
        for k in ('ms', 'flops', 'bytes', 'n', 'floor_cycles'):
            f[k] += d.get(k, 0.0)
    tot_ms = sum(f['ms'] for f in fam.values())
    dom_name, dom = max(fam.items(), key=lambda kv: kv[1]['ms'])
    pk = peaks()
    tensor_bound = dom_name in ('gemm_tn', 'gemm_wgrad')
    if tensor_bound:
        achieved = dom['flops'] / dom['ms'] / 1e9
        peak, unit = pk['tf_sust'], 'TFLOP/s'
    else:
        achieved = dom['bytes'] / dom['ms'] / 1e6
        peak, unit = pk['hbm'], 'GB/s'
    # DRAM traffic of the dominant kernel: per-launch dram read+write bytes of an `ncu --set full` capture of this same
    # command (profiles/r*_ncu_step_full.json, written by tools/ncu_summary.py); null when no capture is committed
    traffic, traffic_note = None, None
    fam_kernel = {'gconv': 'gconv_mma_fwd_kernel', 'gconv_wgrad': 'gconv_mma_wgrad_kernel', 'gemm_tn': 'gemm_tn_pair_kernel',
                  'gemm_wgrad': 'gemm_wgrad_persist_kernel', 'ln_bwd': 'ln2_bwd_kernel', 'ln_fwd': 'ln2_fwd_kernel'}
    for ncu_name in ('r2_ncu_step_final.json', 'r2_ncu_step_full.json', 'r1_ncu_step_full.json'):
        ncu_path = os.path.join(ROOT, 'profiles', ncu_name)
        if os.path.exists(ncu_path) and dom_name in fam_kernel:
            nc = json.load(open(ncu_path)).get('kernels', {}).get(fam_kernel[dom_name])
            if nc and 'avg_dram_bytes_per_launch' in nc:
                traffic = nc['avg_dram_bytes_per_launch']
                traffic_note = (f"dram read+write bytes per launch, ncu --set full over {nc['launches']} launches of "
                                f"{fam_kernel[dom_name]} (profiles/{ncu_name})")
                break
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    mhz = (clocks or {}).get('sm_mhz') or 1965.0
    floor_ms = dom['floor_cycles'] / sms / mhz / 1e3 if dom.get('floor_cycles') else None
    return {'kernel': dom_name, 'bound': 'tensor' if tensor_bound else 'hbm', 'achieved': achieved, 'peak': peak, 'unit': unit,
            'frac': achieved / peak, 'traffic': traffic, 'traffic_note': traffic_note,
            'algorithmic_bytes_per_launch': dom['bytes'] / max(dom['n'], 1), 'algorithmic_flops_per_launch': dom['flops'] / max(dom['n'], 1),
            'peak_source': pk['src'] + (' sustained' if tensor_bound else ''),
            'launches_per_step': dom['n'], 'avg_launch_ms': dom['ms'] / max(dom['n'], 1),
            'share_of_step_kernel_time': dom['ms'] / tot_ms,
            # the grouped-conv kernel is bound by tensor-pipe ISSUE, not by HBM or FLOPs (DESIGN.md 3.1): time of its
            # 3k MMAs per tile at 88 cycles each on every SM at the sampled clock, against the measured time
            'mma_issue_floor': ({'ms': floor_ms, 'frac_of_measured': floor_ms / dom['ms'],
                                 'note': '3k tcgen05.mma (N=48, operands in shared memory, >= 88 cycles each) per 128x48 tile'}
                                if floor_ms else None),
            'families': {k: {'ms': round(v['ms'], 4), 'n': v['n'],
                             'tflops': round(v['flops'] / v['ms'] / 1e9, 1) if v['ms'] else 0,
                             'gbs': round(v['bytes'] / v['ms'] / 1e6, 0) if v['ms'] else 0} for k, v in fam.items()}}


if __name__ == '__main__':
    main()
