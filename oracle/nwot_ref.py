"""fp64 CPU restatement of the NASWOT proxy (`nwot` of nb_asr_b200/proxies.py) on the functions of oracle/model_ref.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The encoder is run exactly as model_ref.forward runs it (dropout off); at
every ReLU20 -- the time-reduction conv of each block and every non-`zero` node op, in module order -- the pre-activation
z (bias included) gives the unit codes m = (0 < z <= 20).  The LSTM and the classifier hold no ReLU and are not run.
    K[i, j] = sum_layers sum_{t < min(L_i, L_j)} sum_c [m_i(t, c) == m_j(t, c)],  L = min(T_k, ceil(audio_len / 2^s_k))
built in numpy as A A^T + B B^T with A = valid * m, B = valid * (1 - m) (exact integers in fp64); score log|det K|.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import model_ref as M


def gate_codes(sd, arch_vec, audio):
    """[(block k, codes (B, C, T_k) bool)] of every ReLU20 layer in module order, fp64 forward."""
    names = M.arch_vec_to_names(arch_vec)
    p = {k: v.detach().double() for k, v in sd.items()}
    x = audio.double()
    out = []
    idx = 0
    with torch.no_grad():
        for b in range(4):
            lp, rp = M.pad_rule(8, 1, M.STRIDES[b])
            z = F.conv1d(F.pad(x, (lp, rp)), p[f'model.{idx}.conv.weight'], p[f'model.{idx}.conv.bias'], stride=M.STRIDES[b])
            out.append((b, (z > 0) & (z <= 20)))
            x = M.relu20(z)
            idx += 1
            x = M.layer_norm_ch(x, p[f'model.{idx}.weight'], p[f'model.{idx}.bias'])
            idx += 1
            for _ in range(M.CELLS[b]):
                outs = [x]
                for n, node in enumerate(names):
                    op, branches = node[0], node[1:]
                    src = outs[-1]
                    q = f'model.{idx}.nodes.{n}.op'
                    if op == 'linear':
                        z = F.linear(src.permute(0, 2, 1), p[q + '.linear.weight'], p[q + '.linear.bias']).permute(0, 2, 1)
                    elif op in M.CONV_EDGE:
                        k, d = M.CONV_EDGE[op]
                        lp, rp = M.pad_rule(k, d, 1)
                        z = F.conv1d(F.pad(src, (lp, rp)), p[q + '.conv.weight'], p[q + '.conv.bias'], dilation=d, groups=M.GROUPS)
                    else:
                        z = None
                    if z is not None:
                        out.append((b, (z > 0) & (z <= 20)))
                        y = M.relu20(z)
                    else:
                        y = torch.zeros_like(src)
                    acc = y
                    for i, bit in enumerate(branches):
                        acc = acc + (outs[i] if bit else torch.zeros_like(outs[i]))
                    outs.append(acc)
                x = M.layer_norm_ch(outs[-1], p[f'model.{idx}.norm_layer.weight'], p[f'model.{idx}.norm_layer.bias'])
                idx += 1
    return out


def frames(audio_len, T_k, k):
    """valid frames of block k: min(T_k, ceil(audio_len / 2^s_k)), s = (0, 0, 1, 2)"""
    s = sum(1 for st in M.STRIDES[:k + 1] if st == 2)
    return np.minimum(T_k, -(-np.asarray(audio_len, np.int64) // (1 << s)))


def kernel_from_codes(codes, audio_len):
    """K (B, B) float64 (exact integers) from [(block k, codes (B, C, T_k) bool)]."""
    B = codes[0][1].shape[0]
    K = np.zeros((B, B), np.float64)
    for k, m in codes:
        m = np.asarray(m, bool)
        T_k = m.shape[2]
        valid = (np.arange(T_k)[None, :] < frames(audio_len, T_k, k)[:, None])[:, None, :]     # (B, 1, T_k)
        a = (m & valid).reshape(B, -1).astype(np.float64)
        b = (~m & valid).reshape(B, -1).astype(np.float64)
        K += a @ a.T + b @ b.T
    return K


def nwot_kernel(sd, arch_vec, audio, audio_len):
    return kernel_from_codes(gate_codes(sd, arch_vec, audio), audio_len)


def nwot_score(K):
    return float(np.linalg.slogdet(np.asarray(K, np.float64))[1])
