"""Static proof, from the SHIPPED library, that the hot kernels are tcgen05 / TMA kernels and that the MMA issue loops are
warp-uniform (round 2, DESIGN.md 3.2): inside `if (lane == 0)` ptxas wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST
sequence of ~20 instructions; in uniform control flow consecutive MMAs are 1-2 instructions apart.  Needs cuobjdump (CUDA
toolkit); runs without a GPU."""
import collections
import re
import shutil
import subprocess

import pytest

from nb_asr_b200 import _build

CUOBJDUMP = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'

# kernel name fragment -> mnemonics that must appear in its SASS
EXPECT = {
    'gemm_tn_pair_kernelILb1': ['UTCHMMA', 'UTMALDG', 'UTMASTG', 'LDTM', 'UTCBAR'],      # staged epilogue: TMA loads and stores
    'gemm_tn_pair_kernelILb0': ['UTCHMMA', 'UTMALDG', 'LDTM', 'UTCBAR'],
    'gemm_wgrad_persist_kernel': ['UTCHMMA', 'UTMALDG', 'LDTM', 'UTCBAR'],
    'gconv_mma_fwd_kernel': ['UTCHMMA', 'UTMALDG', 'UTMASTG', 'LDTM'],
    'gconv_mma_wgrad_kernel': ['UTCHMMA', 'UTMALDG', 'LDTM'],
    'lstm_cluster_fwd_kernelILb1': ['UTCHMMA', 'UTMALDG', 'STTM', 'LDTM', 'UBLKCP'],   # W slice in tensor memory, DSMEM bulk copies
    'lstm_cluster_bwd_kernel': ['UTCHMMA', 'UTMALDG', 'STTM', 'LDTM', 'UBLKCP'],
}


@pytest.fixture(scope='module')
def sass():
    try:
        out = subprocess.run([CUOBJDUMP, '-sass', _build.LIB], capture_output=True, text=True, timeout=600)
    except (OSError, subprocess.TimeoutExpired) as e:
        pytest.skip(f'cuobjdump not usable: {e}')
    if out.returncode != 0 or 'Function :' not in out.stdout:
        pytest.skip('cuobjdump produced no SASS')
    funcs = {}
    for chunk in re.split(r'\n\s*Function : ', out.stdout)[1:]:
        name, body = chunk.split('\n', 1)
        funcs[name.strip()] = [m.group(1) for m in re.finditer(r'/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)', body)]
    return funcs


def _find(funcs, frag):
    hits = [k for k in funcs if frag in k]
    assert len(hits) == 1, (frag, hits)
    return funcs[hits[0]]


@pytest.mark.parametrize('frag', sorted(EXPECT))
def test_hot_kernels_are_tcgen05_tma_kernels(sass, frag):
    ops = collections.Counter(o.split('.')[0] for o in _find(sass, frag))
    for mnem in EXPECT[frag]:
        assert ops[mnem] > 0, (frag, mnem, dict(ops))
    assert ops['HMMA'] == 0, 'no mma.sync fallback inside a tcgen05 kernel'


@pytest.mark.parametrize('frag', sorted(EXPECT))
def test_mma_issue_loops_are_warp_uniform(sass, frag):
    """consecutive tcgen05.mma of an unrolled K loop are at most 3 instructions apart (one uniform add + the MMA); the
    `if (lane == 0)` form needs ~20 (ELECT, 5 x R2UR.BROADCAST, descriptor arithmetic in vector registers)."""
    ops = _find(sass, frag)
    pos = [i for i, o in enumerate(ops) if o.startswith('UTCHMMA')]
    assert len(pos) >= 4
    gaps = sorted(b - a for a, b in zip(pos, pos[1:]))
    assert gaps[len(gaps) // 2] <= 3, (frag, gaps)       # the median gap: loop-carried code between K blocks may be longer
    between = [o for a, b in zip(pos, pos[1:]) if b - a <= 8 for o in ops[a + 1:b]]
    assert not any(o.startswith('R2UR') or o.startswith('ELECT') for o in between), (frag, collections.Counter(between))


def test_no_library_gemm_or_triton_in_the_product_library(sass):
    names = ' '.join(sass)
    assert 'cutlass' not in names.lower() and 'cublas' not in names.lower() and 'triton' not in names.lower()
