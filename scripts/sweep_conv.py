"""Time every tensor-core layer shape of the step (fwd / dgrad / wgrad) with CUDA events.
usage: python scripts/sweep_conv.py [batch]"""
import ctypes as C
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
import vae_gan_b200.functional as VF
from vae_gan_b200 import _lib

dev = torch.device("cuda", 0)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
g = torch.Generator().manual_seed(0)
SHAPES = [  # name, cin, cout, h, k, stride, pad, transposed, count per step (fwd)
    ("G 64->64 s1 @96", 64, 64, 96, 3, 1, 1, False),
    ("G/D 64->128 s2|s1 @96", 64, 128, 96, 3, 1, 1, False),
    ("D 128->128 s1 @96", 128, 128, 96, 3, 1, 1, False),
    ("D 128->256 s2 @96", 128, 256, 96, 3, 2, 1, False),
    ("G 128->128 s1 @48", 128, 128, 48, 3, 1, 1, False),
    ("D 256->256 s1 @48", 256, 256, 48, 3, 1, 1, False),
    ("D 256->512 s2 @48", 256, 512, 48, 3, 2, 1, False),
    ("G 256->256 s1 @24", 256, 256, 24, 3, 1, 1, False),
    ("D 512->512 s1 @24", 512, 512, 24, 3, 1, 1, False),
    ("G convT 256->128 @24", 256, 128, 24, 4, 2, 1, True),
    ("G convT 128->64 @48", 128, 64, 48, 4, 2, 1, True),
    ("D 1x1 128->256 s2 @96", 128, 256, 96, 1, 2, 0, False),
]

def timeit(fn, iters=8):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in evs)
    return sum(ts[1:-1]) / (len(ts) - 2)

print(f"batch {B}")
tot = {"fwd": 0.0, "fwd+stats": 0.0, "dgrad": 0.0, "wgrad": 0.0}
for name, cin, cout, h, k, st, pad, tr in SHAPES:
    geom = VF.ConvGeom(k, st, pad, tr)
    x = VF.as_act(torch.randn(B, cin, h, h, generator=g).to(dev), torch.bfloat16)
    w = (torch.randn((cin, cout, k, k) if tr else (cout, cin, k, k), generator=g) / (cin * k * k) ** 0.5).to(dev)
    d, ho, wo = VF._conv_desc(x.shape, cout, geom, torch.bfloat16, torch.bfloat16)
    pk = torch.empty(w.numel(), dtype=torch.bfloat16, device=dev); pn = torch.empty_like(pk)
    s = _lib.stream_ptr()
    _lib.call("vg_conv_pack_weights", C.byref(d), w.data_ptr(), None, pk.data_ptr(), pn.data_ptr(), s)
    y = VF.empty_act(B, cout, ho, wo, torch.bfloat16, dev)
    dy = VF.as_act(torch.randn(B, cout, ho, wo, generator=g).to(dev), torch.bfloat16)
    dx = torch.empty_like(x)
    dw = torch.zeros_like(w)
    wsb = torch.empty(w.numel(), dtype=torch.float32, device=dev)
    flops = 2.0 * B * (h * h if tr else ho * wo) * cin * cout * k * k
    t_f = timeit(lambda: _lib.call("vg_conv_forward", C.byref(d), x.data_ptr(), pk.data_ptr(), pn.data_ptr(), None, None, y.data_ptr(), None, s))
    st = torch.zeros(2 * cout, dtype=torch.float64, device=dev)
    t_fs = timeit(lambda: _lib.call("vg_conv_forward", C.byref(d), x.data_ptr(), pk.data_ptr(), pn.data_ptr(), None, None, y.data_ptr(), st.data_ptr(), s))
    t_d = timeit(lambda: _lib.call("vg_conv_dgrad", C.byref(d), dy.data_ptr(), pk.data_ptr(), pn.data_ptr(), dx.data_ptr(), s))
    t_w = timeit(lambda: _lib.call("vg_conv_wgrad", C.byref(d), x.data_ptr(), dy.data_ptr(), dw.data_ptr(), None, wsb.data_ptr(), s))
    tot["fwd"] += t_f; tot["fwd+stats"] += t_fs; tot["dgrad"] += t_d; tot["wgrad"] += t_w
    print(f"{name:26s} {flops/1e9:7.1f} GF  fwd {t_f*1e3:7.1f} us {flops/t_f/1e9:7.0f} TF/s (+BN stats {t_fs*1e3:7.1f} us) | dgrad {t_d*1e3:7.1f} us {flops/t_d/1e9:7.0f} | wgrad {t_w*1e3:7.1f} us {flops/t_w/1e9:7.0f}")
print("sum ms", {k: round(v, 3) for k, v in tot.items()})
