"""CPU: host side of the zero-cost proxies -- corrcoef from (Gram, row sums), the scored-tensor rule against the oracle's
module order, the sweep's --proxies flag and the C-ABI table of the proxy kernels."""
import numpy as np
import pytest
import torch

from nb_asr_b200 import _lib, proxies, sweep
from nb_asr_b200.model import ASRModel
from nb_asr_b200 import search_space as ss
from oracle import proxies_ref as R

ARCHS = [[[1, 0], [1, 0, 0], [1, 0, 0, 0]], [[0, 1], [0, 1, 1], [0, 1, 1, 1]], [[5, 1], [1, 1, 0], [5, 0, 1, 1]],
         [[2, 1], [3, 0, 1], [0, 1, 0, 1]], [[5, 0], [5, 0, 0], [5, 0, 0, 0]]]


@pytest.mark.parametrize('B,D', [(2, 7), (8, 1600), (64, 4000)])
def test_corrcoef_from_gram_matches_numpy(B, D):
    rng = np.random.default_rng(B * 1000 + D)
    X = rng.standard_normal((B, D)) * rng.uniform(1e-3, 1e3, (B, 1)) + rng.standard_normal((B, 1))
    c = proxies.corrcoef_from_gram(X @ X.T, X.sum(1), D)
    np.testing.assert_allclose(c, np.corrcoef(X), rtol=0, atol=1e-9)
    assert proxies.jacob_cov_score(c) == pytest.approx(R.jacob_cov_score(np.corrcoef(X)), rel=1e-9)


def test_zero_variance_row_scores_nan():
    X = np.random.default_rng(0).standard_normal((4, 50))
    X[2] = 3.0
    c = proxies.corrcoef_from_gram(X @ X.T, X.sum(1), 50)
    assert np.isnan(proxies.jacob_cov_score(c))


@pytest.mark.parametrize('use_rnn', [True, False])
@pytest.mark.parametrize('arch', ARCHS)
def test_scored_tensors_match_oracle_module_order(arch, use_rnn):
    with torch.device('meta'):
        m = ASRModel(ss.arch_vec_to_names(arch), use_rnn=use_rnn)
    names = proxies.scored_names(m)
    assert names == R.scored_keys(arch, use_rnn)
    params = dict(m.named_parameters())
    assert all(n in params for n in names)
    # excluded: LSTM, LayerNorm, biases
    assert not any('bias' in n or 'norm' in n or '_l0' in n for n in names)


def test_sweep_proxies_flag():
    a = sweep.build_parser().parse_args(['--proxies', 'grad_norm,snip,synflow,jacob_cov', '--proxy-batches', '3'])
    assert a.proxies == ('grad_norm', 'snip', 'synflow', 'jacob_cov') and a.proxy_batches == 3
    a = sweep.build_parser().parse_args(['--proxies', ' jacob_cov '])
    assert a.proxies == ('jacob_cov',) and a.proxy_batches == 1
    a = sweep.build_parser().parse_args([])
    assert a.proxies == () and a.proxy_batches == 1
    for bad in ('fisher', 'snip,grasp', ''):
        with pytest.raises(SystemExit):
            sweep.build_parser().parse_args(['--proxies', bad])


def test_lib_table_has_the_proxy_kernels():
    for n in ('nbasr_transpose_out', 'nbasr_param_stats', 'nbasr_row_gram'):
        assert n in _lib.EXPORTS
