"""CPU: host side of the ZiCo proxy (`zico`) -- the numpy statistic against the official `caculate_zico` transcription
(planted ties, all-zero parameters, a tensor with nothing included), the interleaved split rule, the split-count range,
the --proxies flag and zico's absence from the default measures."""
import numpy as np
import pytest
import torch

from nb_asr_b200 import _lib, proxies, sweep
from oracle import zico_ref as Z


def planted(rng, N, P, scale):
    """(N, P) fp32-valued samples: random columns, columns of N equal values, all-zero columns"""
    G = (rng.standard_normal((N, P)) * scale).astype(np.float32)
    G[:, 3::7] = G[0, 3::7]                          # all equal: std exactly 0
    G[:, 5::11] = 0.0                                # all zero
    G[1:, 2::13] = G[0, 2::13]                       # equal except the first sample: included
    return G.astype(np.float64)


@pytest.mark.parametrize('N', [2, 3, 8])
def test_statistic_equals_official_transcription(N):
    rng = np.random.default_rng(N)
    grads = {'a': planted(rng, N, 1000, 1.0), 'b': planted(rng, N, 77, 1e-30), 'c': planted(rng, N, 5, 1e3)}
    # nothing included (fp32 values: N equal fp64 values with more than 24 significant bits need not sum exactly)
    grads['tied'] = np.repeat(rng.standard_normal((1, 40)).astype(np.float32), N, axis=0).astype(np.float64)
    grads['zero'] = np.zeros((N, 9))
    layers = Z.zico_layers(grads)
    assert set(layers) == {'a', 'b', 'c'}                                   # skipped, not -inf
    official = Z.caculate_zico({k: v.copy() for k, v in grads.items()})
    assert np.isfinite(official)
    assert sum(layers.values()) == pytest.approx(official, rel=1e-13, abs=0)
    for k in ('a', 'b', 'c'):
        G = grads[k]
        R, n = Z.snr_stats(G)
        std = np.std(G, axis=0)
        assert n == np.count_nonzero(std) == np.count_nonzero(np.any(G != G[0], axis=0))
        assert np.log(R) == pytest.approx(Z.caculate_zico({k: G.copy()}), rel=1e-13)
    assert Z.snr_stats(grads['tied']) == (0.0, 0) and Z.snr_stats(grads['zero']) == (0.0, 0)


def test_split_rule_interleaves_and_keeps_T():
    B, T = 7, 11
    audio = torch.arange(B, dtype=torch.float32)[:, None, None].expand(B, 80, T).clone()
    alen = torch.arange(10, 10 + B)
    tg = torch.arange(B, dtype=torch.int32)[:, None].expand(B, 4).clone()
    tl = torch.arange(1, 1 + B)
    for N in (2, 3, 7):
        parts = proxies.zico_split(((audio, alen), (tg, tl)), N)
        assert len(parts) == N
        for k, ((a, al), (t, tl_)) in enumerate(parts):
            idx = list(range(k, B, N))
            assert a.shape[1:] == (80, T) and a[:, 0, 0].tolist() == idx
            assert al.tolist() == [10 + i for i in idx] and t[:, 0].tolist() == idx and tl_.tolist() == [1 + i for i in idx]


@pytest.mark.parametrize('B,N', [(8, 1), (8, 0), (8, 9), (4, 5), (64, 17), (2, 3)])
def test_split_count_out_of_range_raises(B, N):
    batch = ((torch.zeros(B, 80, 5), torch.full((B,), 5)), (torch.ones(B, 2, dtype=torch.int32), torch.full((B,), 2)))
    with pytest.raises(ValueError):
        proxies.zico_split(batch, N)
    with pytest.raises(ValueError):
        proxies.compute_proxies(None, batch, ('zico',), zico_splits=N)         # before the model is touched


def test_split_count_bounds_accepted():
    for B, N in ((2, 2), (64, 16), (16, 16)):
        batch = ((torch.zeros(B, 80, 5), torch.full((B,), 5)), (torch.ones(B, 2, dtype=torch.int32), torch.full((B,), 2)))
        assert len(proxies.zico_split(batch, N)) == N


def test_zico_is_accepted_by_name_but_not_a_default():
    assert 'zico' not in proxies.MEASURES
    assert proxies.MEASURES == ('grad_norm', 'snip', 'synflow', 'jacob_cov', 'nwot')
    assert proxies.parse_measures('zico') == ('zico',)
    assert proxies.parse_measures('grad_norm, zico') == ('grad_norm', 'zico')
    with pytest.raises(ValueError):
        proxies.parse_measures('zico,fisher')
    assert sweep.build_parser().parse_args(['--proxies', 'zico']).proxies == ('zico',)
    assert sweep.build_parser().parse_args(['--proxies', 'nwot,zico']).proxies == ('nwot', 'zico')
    assert 'zico' in sweep.build_parser().format_help()


def test_lib_table_has_grad_snr():
    assert 'nbasr_grad_snr' in _lib.EXPORTS
