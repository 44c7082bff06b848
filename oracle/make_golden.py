"""Generate tests/golden/* by running the REAL reference (/root/reference) on CPU.

Run in the build container only (the reference does not travel to the GPU box):
    python oracle/make_golden.py
The reference code is imported unmodified behind four shims (SURVEY.md §8c):
  1. torchaudio.set_audio_backend no-op      (training/torch/timit.py:11)
  2. stub module torch_edit_distance         (training/torch/trainer.py:8)
  3. stub module ctcdecode.CTCBeamDecoder    (training/torch/trainer.py:9,71)
  4. torch.clamp_max_ -> out-of-place        (model/torch/ops.py:28,47 break autograd on torch>=1.8)
"""
import hashlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = os.environ.get('NBASR_REFERENCE', '/root/reference')
GOLD = os.path.join(ROOT, 'tests', 'golden')


def import_reference():
    from oracle.reference_shims import import_reference as _imp
    nasbench_asr = _imp(REF)
    from nasbench_asr.training.torch.encoder import PhonemeEncoder
    return nasbench_asr, PhonemeEncoder


def digest(sd):
    h = hashlib.sha256()
    for k in sd:
        h.update(k.encode())
        h.update(sd[k].detach().contiguous().numpy().tobytes())
    return h.hexdigest()


def summarize(tensors):
    out = {}
    for k, v in tensors.items():
        f = v.detach().double().flatten()
        out[k] = dict(norm=float(f.norm()), sum=float(f.sum()), head=[float(x) for x in f[:8]],
                      shape=list(v.shape))
    return out


ARCHS = {
    'default': [[1, 0], [1, 0, 0], [1, 0, 0, 0]],
    'c7d2_skips': [[4, 1], [4, 1, 1], [4, 1, 1, 1]],
    'linear_skips': [[0, 1], [0, 1, 1], [0, 1, 1, 1]],
    'mixed': [[2, 1], [3, 0, 1], [0, 1, 0, 1]],
    'zero_mix': [[5, 1], [1, 1, 0], [5, 0, 1, 1]],
    'c5_c7': [[1, 1], [3, 1, 0], [2, 0, 0, 1]],
}


def main():
    from oracle import model_ref as M
    nb, PhonemeEncoder = import_reference()
    os.makedirs(GOLD, exist_ok=True)
    enc = PhonemeEncoder(48)
    meta = {}

    # fold LUT (encoder.py:64-74), effective chained table over classes 0..48
    x = torch.arange(49, dtype=torch.int32)
    lut = enc.fold_encoded(x.clone(), 39).tolist()
    json.dump(dict(lut=lut, idx_mapping={int(k): int(v) for k, v in enc.idx_mappings[1][2].items()},
                   vocab48=enc.get_vocab(inc_blank=True)),
              open(os.path.join(GOLD, 'fold_lut.json'), 'w'))

    def ref_trainer(model):
        tr = nb.get_trainer((enc, None, None, None), nb.get_loss(), gpus=[], save_dir=None, verbose=False)
        tr.model = tr._model = model
        tr.optimizer = torch.optim.Adam(model.parameters(), lr=1e-4, eps=1e-7)
        return tr

    # ---- eval fixtures: survey fixture B=8,T=500 (4 archs) and small B=3,T=70 (all archs)
    for tag, (B, T), names in (('survey', (8, 500), ['default', 'c7d2_skips', 'linear_skips', 'mixed']),
                               ('small', (3, 70), list(ARCHS))):
        batch = M.make_batch(B, T, seed=0, min_len=T // 2)
        audio, alen, targets, tl = batch
        for name in names:
            arch = ARCHS[name]
            nb.set_seed(1235)
            model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0)
            model.eval()
            tr = ref_trainer(model)
            with torch.no_grad():
                logits = model(audio)
            loss, logp, out_len = tr.step(((audio, alen), (targets.clone(), tl)), training=False)
            key = f'{tag}_{name}'
            np.savez_compressed(os.path.join(GOLD, f'eval_{key}.npz'),
                                logits=logits.numpy(), loss=np.float32(loss.item()),
                                out_len=out_len.numpy(), logp_sum=np.float64(logp.double().sum().item()))
            meta[key] = dict(arch=arch, B=B, T=T, sd_digest=digest(model.state_dict()),
                             n_params=sum(p.numel() for p in model.parameters()),
                             loss=float(loss.item()))
            print(key, meta[key]['loss'], meta[key]['n_params'], flush=True)

    # ---- train fixtures: two consecutive reference Trainer.step(training=True) calls
    B, T = 3, 70
    audio, alen, targets, tl = M.make_batch(B, T, seed=0, min_len=T // 2)
    for name in ARCHS:
        arch = ARCHS[name]
        nb.set_seed(1235)
        model = nb.get_model(arch, use_rnn=True, dropout_rate=0.0)
        model.train()
        tr = ref_trainer(model)
        rec = {}
        for it in range(2):
            loss, logp, _ = tr.step(((audio, alen), (targets.clone(), tl)), training=True)
            rec[f'loss{it}'] = float(loss.item())
            if it == 0:
                # grads after clip_grad_norm_ (in place) of step 0, and the parameters after its update; the tests
                # compare the second step through loss1 only (meta.json stays under 1 MB)
                rec['grads_clipped'] = summarize({k: p.grad for k, p in model.named_parameters()})
                rec['params0'] = summarize(dict(model.named_parameters()))
        meta[f'train_{name}'] = dict(arch=arch, B=B, T=T, **rec)
        print('train', name, rec['loss0'], rec['loss1'], flush=True)

    # infeasible-alignment fixture (zero_infinity): target longer than output_len
    nb.set_seed(1235)
    lp = torch.log_softmax(torch.randn(2, 6, 49, generator=torch.Generator().manual_seed(3)), dim=2)
    tg = torch.randint(1, 49, (2, 9), generator=torch.Generator().manual_seed(4), dtype=torch.int32)
    loss = nb.get_loss()(lp, torch.tensor([6, 6]), tg, torch.tensor([9, 3]))
    np.savez_compressed(os.path.join(GOLD, 'ctc_infeasible.npz'), logp=lp.numpy(), targets=tg.numpy(),
                        out_len=np.array([6, 6]), tgt_len=np.array([9, 3]), loss=np.float32(loss.item()))

    json.dump(meta, open(os.path.join(GOLD, 'meta.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
