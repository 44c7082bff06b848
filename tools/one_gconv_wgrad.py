"""Time the grouped-conv weight-gradient kernel on the bench shapes (64 x 500, C = 600 .. 1200 or $C), with the activation
read as a bf16 copy (nbasr_gconv_wgrad) and as the forward's scaled fp16 tensor (nbasr_gconv_wgrad_x, x_scale = 1/32; skipped
on a library without it).  L2 is overwritten between launches."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from nb_asr_b200 import _lib
from nb_asr_b200._lib import BF16, F16
import gpu_utils as U
lib = _lib.load()
has_x = hasattr(lib, 'nbasr_gconv_wgrad_x')
B, T, k, d = 64, int(os.environ.get('T', 500)), int(os.environ.get('K', 5)), int(os.environ.get('D', 1))
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=U.DEV)
for Cc in ([int(os.environ['C'])] if 'C' in os.environ else [600, 800, 1000, 1200]):
    cpg = Cc // 100
    xt = torch.randn(B, T, Cc)
    xs = {'bf16': U.to_padded(xt, BF16), 'fp16': U.to_padded(xt * 32, F16)}
    dz = U.to_padded(torch.randn(B, T, Cc), BF16)
    dw = torch.zeros(Cc, cpg, k, device=U.DEV)
    db = torch.zeros(Cc, device=U.DEV)
    for with_bias in (1, 0):
        for fmt in ('bf16', 'fp16') if has_x else ('bf16',):
            x = xs[fmt]
            ts = []
            for it in range(12):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                args = (B, T, U.geo(T), Cc, cpg, k, 0 if d == 1 else -8, d, dw.data_ptr(), db.data_ptr() if with_bias else None, U.stream())
                if fmt == 'bf16':
                    _lib.check(lib.nbasr_gconv_wgrad(BF16, dz.data_ptr(), x.data_ptr(), *args))
                else:
                    _lib.check(lib.nbasr_gconv_wgrad_x(BF16, dz.data_ptr(), x.data_ptr(), F16, 1.0 / 32, *args))
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ts = sorted(ts[2:])
            t = ts[len(ts) // 2]
            print(f'C={Cc} T={T} k={k} d={d} wgrad x={fmt} bias={with_bias}: {t*1e3:7.1f} us (min {ts[0]*1e3:.1f}, max {ts[-1]*1e3:.1f})'
                  f'  {2*B*T*Cc*2/t/1e6:6.0f} GB/s (dz + x read once)', flush=True)
