"""Architecture-sharded sweep evaluation (BASELINE.json configs[3]): every candidate arch_vec is built from the
same seed, run through the eval step (forward + CTC loss + greedy decode + PER) on a fixed synthetic set and
reported as one row.  Candidates are independent: rank r evaluates its shard (nb_asr_b200.distributed.shard_archs),
no collective touches the data path, rows are gathered on rank 0.

    torchrun --nproc-per-node 8 -m nb_asr_b200.sweep --limit 0          # all 8 242 unique candidates on 8 GPUs
The reference has no sweep driver (SURVEY.md §3.5); enumeration follows search_space.get_all_architectures and, by
default, keeps the first arch_vec of every graph-isomorphism class (graph_utils.get_model_hash: 13 824 -> 8 242).
``--out-pickle`` writes an nb-asr style table (README "Dataset format": pickle.dump(header) then pickle.dump(rows),
row order = header['columns']).
"""
import argparse
import json
import os
import time

import torch

import pickle

from . import PhonemeEncoder, data, distributed, get_loss, get_model, get_trainer, graph_utils, search_space, set_seed


def evaluate_arch(arch, batches, gpu, precision='bf16', seed=1235, init='reference', conv_gain=1.0, n_ref=None, proxies=(),
                  proxy_batches=1):
    """One candidate: build from `seed`, eval step (forward + CTC loss) and greedy decode + PER on every batch.
    Returns the reference's epoch metrics (AvgMeter, trainer.py:16-33: unweighted mean of the per-batch means) plus the
    corpus-level PER (sum of edit distances / sum of reference lengths), and for every measure in `proxies` its
    zero-cost proxy score (nb_asr_b200.proxies) averaged over the first `proxy_batches` batches."""
    if init == 'reference':
        set_seed(seed)
    model = get_model(arch, use_rnn=True, dropout_rate=0.0, gpu=gpu, precision=precision, init=init, seed=seed, conv_gain=conv_gain)
    model.eval()
    model.engine.max_plans = 64                    # one inference plan per padded length of the evaluation set
    tr = get_trainer((PhonemeEncoder(48), None, None, None), get_loss(), gpus=[gpu], verbose=False)
    tr.model = tr._model = model
    losses, pers, dists = [], [], []
    for batch in batches:
        loss, logp, out_len = tr.step(batch, training=False)
        per = tr.decode(logp, out_len, batch)
        losses.append(loss.double())
        pers.append(per.double())
        dists.append(tr.last_hyp[2].sum().double())
    res = torch.stack([torch.stack(losses).mean(), torch.stack(pers).mean(), torch.stack(dists).sum()]).tolist()
    scores = {}
    if proxies:
        from .proxies import compute_proxies
        use = batches[:max(1, proxy_batches)]
        per_batch = [compute_proxies(model, b, proxies) for b in use]
        scores = {m: sum(p[m] for p in per_batch) / len(per_batch) for m in proxies}
    model._engine = None
    row = dict(arch=arch, loss=res[0], per=res[1])
    if n_ref:
        row['per_corpus'] = res[2] / n_ref
    row.update(scores)
    return row


def proxy_list(text):
    """argparse type of --proxies: comma-separated measure names of nb_asr_b200.proxies.MEASURES."""
    from .proxies import parse_measures
    try:
        return parse_measures(text)
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e)) from e


def build_parser():
    ap = argparse.ArgumentParser()


    ap.add_argument('--limit', type=int, default=16, help='number of architectures (0 = the whole list)')
    ap.add_argument('--arch-file', default=None, help='JSON list of arch_vecs (e.g. the 8242 unique ones)')
    ap.add_argument('--dataset', default='timit', choices=['timit', 'uniform'],
                    help="timit: the fixed 1344-utterance TIMIT-shaped set of BASELINE.json configs[3]; uniform: --n-batches x --batch x --frames")
    ap.add_argument('--utterances', type=int, default=1344)
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--frames', type=int, default=320)
    ap.add_argument('--n-batches', type=int, default=2)
    ap.add_argument('--precision', default='bf16')
    ap.add_argument('--init', default='device', choices=['device', 'reference'],
                    help='device: weights drawn on the GPU (same distributions as the reference init, milliseconds); '
                         'reference: the reference procedure on the host RNG (same-seed bit-identical weights, 0.3-1.1 s per arch)')
    ap.add_argument('--conv-gain', type=float, default=101 ** 0.5,
                    help='multiplier of the xavier bound of the grouped-conv edges (device init only); sqrt(1 + groups) makes '
                         'them variance-preserving so that skip-free conv archs do not decode all-blank (SURVEY finding 5)')
    ap.add_argument('--seed', type=int, default=1235)
    ap.add_argument('--balance', default='lpt', choices=['lpt', 'rr'])
    ap.add_argument('--out', default=None)
    ap.add_argument('--out-pickle', default=None, help='nb-asr style table: header, then rows')
    ap.add_argument('--all', action='store_true', help='evaluate every arch_vec, not one per isomorphism class')
    ap.add_argument('--proxies', type=proxy_list, default=(),
                    help='comma-separated zero-cost proxies to add as columns: grad_norm,snip,synflow,jacob_cov,nwot')
    ap.add_argument('--proxy-batches', type=int, default=1,
                    help='the proxies are averaged over the first N batches of the evaluation set')
    return ap


def main():
    args = build_parser().parse_args()
    if args.proxy_batches < 1:
        raise SystemExit('--proxy-batches must be >= 1')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    # Ranks map round-robin onto the visible GPUs; more ranks than GPUs is allowed: a candidate costs host time (module
    # tree, plans for every padded length) besides its GPU time, so two processes per GPU keep it busy.  Rows are only
    # gathered at the end -> gloo, no NCCL communicator needed: the data path has no collective.
    n_gpus = max(1, torch.cuda.device_count())
    local = local % n_gpus
    torch.cuda.set_device(local)
    if world > 1:
        torch.distributed.init_process_group('gloo')
    if args.arch_file:
        archs = json.load(open(args.arch_file))
    elif args.all:
        archs = list(search_space.get_all_architectures())
    else:
        archs = [a for _, a in graph_utils.get_unique_architectures()]
    archs = archs[:args.limit] if args.limit else archs
    if args.dataset == 'timit':
        batches = data.timit_shaped_eval_set(n_utt=args.utterances, batch_size=args.batch, seed=0)
    else:
        batches = [data.make_batch(args.batch, args.frames, seed=100 + i, min_len=args.frames // 3) for i in range(args.n_batches)]
    mean_frames = sum(float(al.sum()) for (a, al), _ in batches) / sum(al.numel() for (a, al), _ in batches)
    mine = distributed.shard_archs(archs, rank, world, balance=args.balance, frames=int(mean_frames))
    n_ref = sum(int(tl.sum()) for _, (t, tl) in batches)
    dev = torch.device('cuda', local)
    batches = [((a.to(dev), al.to(dev)), (t.to(dev), tl.to(dev))) for (a, al), (t, tl) in batches]
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t0 = time.time()
    rows = []
    for i in mine:
        r = evaluate_arch(archs[i], batches, local, args.precision, seed=args.seed, init=args.init, conv_gain=args.conv_gain, n_ref=n_ref,
                          proxies=args.proxies, proxy_batches=args.proxy_batches)
        r['index'] = i
        r['hash'] = graph_utils.get_model_hash(archs[i])
        rows.append(r)
    torch.cuda.synchronize()
    dt = time.time() - t0
    if world > 1:
        tt = torch.tensor([dt], dtype=torch.float64)
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)      # the sweep ends with its slowest rank
        dt = float(tt.item())
    rows = distributed.gather_rows(rows)
    if rank == 0:
        rows.sort(key=lambda r: r['index'])
        n_utt = sum(al.numel() for (a, al), _ in batches)
        audio_s = sum(float(al.sum()) for (a, al), _ in batches) / 100.0 * len(archs)
        pers = [r['per'] for r in rows]
        summary = dict(n_archs=len(archs), world=world, gpus=min(world, n_gpus), seconds=dt, archs_per_s=len(archs) / dt,
                       audio_s_per_s=audio_s / dt, utterances_per_arch=n_utt, dataset=args.dataset, init=args.init,
                       conv_gain=args.conv_gain if args.init == 'device' else 1.0, precision=args.precision,
                       per_min=min(pers), per_max=max(pers), per_mean=sum(pers) / len(pers),
                       archs_with_trivial_per=sum(1 for p in pers if p == 1.0))
        print(json.dumps(summary))
        if args.out:
            json.dump(dict(summary=summary, rows=rows), open(args.out, 'w'))
        if args.out_pickle:
            header = dict(dataset_type='b200-sweep-eval', version=2, search_space=search_space.get_search_space(),
                          ops=search_space.all_ops, columns=['model_hash', 'arch_vec', 'ctc_loss', 'per', 'per_corpus'] + list(args.proxies),
                          seed=args.seed, precision=args.precision, dataset=args.dataset, utterances=n_utt, init=args.init,
                          conv_gain=summary['conv_gain'], data='synthetic', decode='greedy')
            if args.proxies:
                header['proxy_batches'] = min(args.proxy_batches, len(batches))
            with open(args.out_pickle, 'wb') as f:
                pickle.dump(header, f)
                pickle.dump([[r['hash'], r['arch'], r['loss'], r['per'], r.get('per_corpus')] + [r[m] for m in args.proxies]
                             for r in rows], f)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
