"""-m gpu: the grouped-conv weight gradient reading the forward's scaled fp16 activations (nbasr_gconv_wgrad_x, x_scale = 1/S)
instead of an unscaled bf16 copy of them, on the tcgen05 kernel and on the SIMT kernel, and the 16-bit grad plans that now
write a bf16 twin only for the activations a dense weight gradient reads."""
import os
import re
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import gpu_utils as U  # noqa: E402
import nb_asr_b200 as nb  # noqa: E402
from nb_asr_b200 import _lib  # noqa: E402
from nb_asr_b200._lib import BF16, F16  # noqa: E402
from nb_asr_b200.engine import ACT_SCALE, dense_wgrad_inputs  # noqa: E402
from nb_asr_b200.model import CONV_EDGES, pad_rule  # noqa: E402

S = ACT_SCALE
HERE = os.path.dirname(os.path.abspath(__file__))


def wgrad_errors(cpg, op, bias, seed=0):
    """(error of the fp16-X call, error of the bf16-copy call, larger bias-gradient error of the two), relative to fp64 torch on the true
    activation x and the bf16 gradient dZ.  B * T = 903 is not a multiple of the 128-frame tile."""
    torch.manual_seed(seed)
    Cc, (k, d) = 100 * cpg, CONV_EDGES[op]
    B, T = 3, 301
    lp, _ = pad_rule(k, d, 1)
    # a ReLU20 / LayerNorm-like spread of magnitudes, with some values deep in fp16's subnormal range once scaled
    x = torch.randn(B, T, Cc, dtype=torch.float64) * torch.exp(torch.randn(B, T, Cc, dtype=torch.float64))
    dz = torch.randn(B, T, Cc).bfloat16().double()
    w = torch.zeros(Cc, cpg, k, dtype=torch.float64, requires_grad=True)
    z = F.conv1d(F.pad(x.permute(0, 2, 1), (lp, (k - 1) * d - lp)), w, dilation=d, groups=100).permute(0, 2, 1)
    gw, = torch.autograd.grad(z, w, dz)
    lib = _lib.load()
    xh = U.to_padded((x * S).float(), F16)               # what a 16-bit forward stores
    xb = U.to_padded(x.float(), BF16)                    # the bf16 copy it used to store as well
    dzb = U.to_padded(dz.float(), BF16)
    out = []
    for xbuf, xdt, xs in ((xh, F16, 1.0 / S), (xb, BF16, 1.0)):
        dw = torch.zeros(Cc, cpg, k, device=U.DEV)
        db = torch.zeros(Cc, device=U.DEV) if bias else None
        _lib.check(lib.nbasr_gconv_wgrad_x(BF16, dzb.data_ptr(), xbuf.data_ptr(), xdt, xs, B, T, U.geo(T), Cc, cpg, k, -lp, d,
                                           dw.data_ptr(), db.data_ptr() if bias else None, U.stream()))
        torch.cuda.synchronize()
        out.append(U.relerr(dw.cpu().double(), gw))
        if bias:
            out.append(U.relerr(db.cpu().double(), dz.sum((0, 1))))
    if bias:
        return out[0], out[2], max(out[1], out[3])
    return out[0], out[1], 0.0


@pytest.mark.parametrize('bias', [1, 0])
@pytest.mark.parametrize('op', sorted(CONV_EDGES))
@pytest.mark.parametrize('cpg', [6, 8, 10, 12])
def test_fp16_x_matches_fp64_like_the_bf16_copy(cpg, op, bias):
    e16, eb, edb = wgrad_errors(cpg, op, bias)
    # dZ . bf16(fp16(S x) / S) vs dZ . bf16(x): a fraction of elements rounds twice (<= 1 bf16 ulp), and below |x| ~ 2e-6
    # fp16 holds fewer bits than bf16 -- the same ratio rule as the input-gradient test
    assert e16 <= 1.5 * eb + 1e-7, (e16, eb)
    assert e16 < 1e-2, e16
    assert edb < 1e-4, edb


@pytest.mark.skipif(os.environ.get('NBASR_FORCE_SIMT') == '1', reason='already the SIMT run')
def test_simt_kernel_in_a_subprocess():
    """NBASR_FORCE_SIMT is latched when the library loads: run the same cases in a fresh process"""
    env = dict(os.environ, NBASR_FORCE_SIMT='1')
    r = subprocess.run([sys.executable, '-s', '-m', 'pytest', '-q', '-p', 'no:cacheprovider', os.path.abspath(__file__),
                        '-k', 'test_fp16_x_matches_fp64_like_the_bf16_copy and (conv5d2 or conv7)'],
                       cwd=os.path.dirname(HERE), env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and re.search(r'\b24 passed', r.stdout), r.stdout[-4000:] + r.stderr[-4000:]


DEFAULT = [[1, 0], [1, 0, 0], [1, 0, 0, 0]]


@pytest.mark.parametrize('dropout', [0.0, 0.1])
def test_grad_plan_twins_exactly_the_dense_wgrad_inputs(dropout):
    nb.set_seed(1235)
    model = nb.get_model(DEFAULT, use_rnn=True, dropout_rate=dropout, gpu=0, precision='bf16')
    eng = model.engine
    want = dense_wgrad_inputs(model.arch_desc, model.use_norm, model.use_rnn, input_dropout=dropout > 0)
    pl = eng.plan(4, 120, True)
    assert set(pl.twins) == want
    assert all(t.dtype == torch.bfloat16 for t in pl.twins.values())
    assert eng.plan(4, 120, False, grad=True).twins.keys() == dense_wgrad_inputs(model.arch_desc, True, True)
    assert eng.plan(4, 120, False).twins == {}                         # eval plans: no backward, no twins
    fp32 = nb.get_model(DEFAULT, use_rnn=True, dropout_rate=dropout, gpu=0, precision='fp32')
    assert fp32.engine.plan(4, 120, True).twins == {}                # fp32: the activations are the weight-gradient operand

