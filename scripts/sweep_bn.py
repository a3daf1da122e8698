"""Time the BatchNorm-family kernels on the 128-channel 96x96 tensor (batch 64 = 151 MB) with CUDA events."""
import ctypes as C, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
import vae_gan_b200.functional as VF
from vae_gan_b200 import _lib
dev = torch.device("cuda", 0)
B, Cc, H = 64, int(sys.argv[1]) if len(sys.argv) > 1 else 128, 96
g = torch.Generator().manual_seed(0)
x = VF.as_act(torch.randn(B, Cc, H, H, generator=g).to(dev), torch.bfloat16)
dy = VF.as_act(torch.randn(B, Cc, H, H, generator=g).to(dev), torch.bfloat16)
y = torch.empty_like(x); dx = torch.empty_like(x)
gamma = torch.ones(Cc, device=dev); beta = torch.zeros(Cc, device=dev)
mr = torch.cat([torch.zeros(Cc), torch.ones(Cc)]).to(dev)
sums = torch.zeros(2 * Cc, dtype=torch.float64, device=dev)
d = VF._bn_desc(x, 0.2, 0.0, 0, True)
s = _lib.stream_ptr()
MB = x.numel() * 2 / 1e6
def timeit(fn, iters=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return sum(t[1:-1]) / (len(t) - 2)
cases = {
  "stats (1x)": (1, lambda: _lib.call("vg_bn_stats", x.data_ptr(), C.byref(d), sums.data_ptr(), s)),
  "act_fwd (2x)": (2, lambda: _lib.call("vg_bn_act_forward", x.data_ptr(), mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(), C.byref(d), y.data_ptr(), s)),
  "bwd_reduce (2x)": (2, lambda: _lib.call("vg_bn_act_backward_reduce", dy.data_ptr(), x.data_ptr(), mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(), C.byref(d), sums.data_ptr(), s)),
  "bwd_apply (3x)": (3, lambda: _lib.call("vg_bn_act_backward_apply", dy.data_ptr(), x.data_ptr(), mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(), sums.data_ptr(), float(B*H*H), C.byref(d), None, None, dx.data_ptr(), s)),
  "bn_add+stats (3x)": (3, lambda: _lib.call("vg_bn_add_forward", x.data_ptr(), None, None, None, dy.data_ptr(), mr.data_ptr(), gamma.data_ptr(), beta.data_ptr(), C.byref(d), y.data_ptr(), sums.data_ptr(), s)),
}
print(f"C={Cc} tensor {MB:.0f} MB")
for name, (mult, fn) in cases.items():
    t = timeit(fn)
    print(f"  {name:20s} {t*1e3:7.1f} us  {mult*MB/t/1e3:6.2f} TB/s  {100*mult*MB/t/1e3/6.5389:5.1f}% of measured HBM")
