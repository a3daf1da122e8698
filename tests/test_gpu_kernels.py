"""Per-kernel parity (-m gpu): each C-ABI entry point against plain fp32 torch math / the oracle on
the same seeded inputs.  fp32 path tolerance 1e-5 (max-normalised), bf16 tensor-core path 2e-2 -
the tolerances BASELINE.json north_star states."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vaegan_oracle as O
from tests.gpu_util import assert_close, dev, nchw, philox_keep2d, philox_mask_nchw, relmax

pytestmark = pytest.mark.gpu

TOL32 = 1e-5
TOL16 = 2e-2


@pytest.fixture(scope="module", autouse=True)
def _setup():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    import vae_gan_b200  # noqa: F401  (fails loudly if the .so is missing)
    yield


def VF():
    import vae_gan_b200.functional as vf
    return vf


def rand_act(shape, dtype, seed, scale=1.0, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(shape, generator=g) * scale + shift)
    vf = VF()
    return vf.as_act(x.to(dev()), dtype), x


# ------------------------------------------------------------------------------------------------
def test_library_loads_and_inits():
    from vae_gan_b200 import _lib
    lib = _lib.load()
    assert lib.vg_version() == 100
    _lib.ensure_device(dev())
    assert torch.cuda.get_device_capability(0)[0] == 10


def test_philox_masks_bit_exact():
    vf = VF()
    seed = vf.rng.seed
    for shape, p, off, step, so in [((2, 8, 4, 4), 0.5, 3, None, 0), ((3, 6, 5, 7), 0.3, 11, 2, 0),
                                    ((2, 1, 8, 8), 0.5, 0, None, 5), ((1, 64, 3, 3), 0.9, 70000, 1, 2)]:
        m = vf.export_dropout_mask(shape, p, off, dev(), step=step, sample_offset=so).cpu()
        want = philox_mask_nchw(shape, seed, off, p, step or 0, so)
        assert torch.equal(m.contiguous(), want), (shape, p, off)
    from vae_gan_b200 import _lib
    for n, c, p, off, so in [(4, 16, 0.5, 7, 0), (3, 10, 0.25, 9, 3)]:
        out = torch.empty((n, c), dtype=torch.float32, device=dev())
        _lib.call("vg_dropout2d_scale", out.data_ptr(), n, c, p, seed, off, None, so, _lib.stream_ptr())
        want = torch.from_numpy(O.philox_keep_scale2d(n, c, seed, off, p, sample_offset=so))
        assert torch.equal(out.cpu(), want)


def test_philox_uniform_bit_exact_and_partition_invariant():
    """vg_philox_uniform (gradient-penalty interpolation weights) against the oracle's integer restatement."""
    from vae_gan_b200 import _lib
    seed = 0xABCDEF12345
    for n, off, start in [(7, 3, 0), (64, 65536 * 2 + 5, 0), (33, 9, 16)]:
        out = torch.empty(n, dtype=torch.float32, device=dev())
        _lib.call("vg_philox_uniform", out.data_ptr(), n, seed, off, None, start, _lib.stream_ptr())
        want = torch.from_numpy(O.philox_uniform(n, seed, off, start))
        assert torch.equal(out.cpu(), want)
        assert float(out.min()) >= 0.0 and float(out.max()) < 1.0
    a = torch.empty(32, dtype=torch.float32, device=dev())
    b = torch.empty(16, dtype=torch.float32, device=dev())
    _lib.call("vg_philox_uniform", a.data_ptr(), 32, seed, 4, None, 0, _lib.stream_ptr())
    _lib.call("vg_philox_uniform", b.data_ptr(), 16, seed, 4, None, 16, _lib.stream_ptr())
    assert torch.equal(a[16:], b)          # rank 1 of 2 draws the same numbers for its samples


@pytest.mark.parametrize("c_in,c_out,k,transposed", [(64, 128, 3, False), (128, 64, 4, True), (18432, 1024, 1, False), (100, 72, 3, False),
                                                     (72, 100, 4, True), (40, 200, 1, False), (24, 40, 5, False), (8, 8, 3, False),
                                                     (512, 512, 3, False)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_weight_pack_layouts_bit_exact(c_in, c_out, k, transposed, dtype):
    """vg_conv_pack_weights: both packed layouts ([tap][c_out][c_in] and [tap][c_in][c_out]) are pure permutations
    (+ division by sigma, + cast) of the torch weight - bit-exact against torch, for every kernel variant the
    launcher picks (1x1 transpose, tiled 3x3 / 4x4, element-wise fallback) incl. ragged channel counts."""
    vf = VF()
    from vae_gan_b200 import _lib
    g = torch.Generator().manual_seed(c_in * 7 + c_out + k)
    shape = (c_in, c_out, k, k) if transposed else (c_out, c_in, k, k)
    w = torch.randn(shape, generator=g).to(dev())
    sigma = torch.tensor([1.7], device=dev())
    d, _, _ = vf._conv_desc((1, c_in, 8, 8), c_out, vf.ConvGeom(k, 1, 0 if k == 1 else 1, transposed), dtype, dtype)
    for sg in (None, sigma):
        kn = torch.empty(w.numel(), dtype=dtype, device=dev())
        nk = torch.empty(w.numel(), dtype=dtype, device=dev())
        _lib.call("vg_conv_pack_weights", C.byref(d), w.data_ptr(), sg.data_ptr() if sg is not None else None, kn.data_ptr(), nk.data_ptr(),
                  _lib.stream_ptr())
        ws = (w * (1.0 / sigma)) if sg is not None else w      # the kernels multiply by 1/sigma
        w4 = ws.permute(1, 0, 2, 3) if transposed else ws      # -> [c_out][c_in][kh][kw]
        want_kn = w4.permute(2, 3, 0, 1).reshape(-1).to(dtype)  # [tap][c_out][c_in]
        want_nk = w4.permute(2, 3, 1, 0).reshape(-1).to(dtype)  # [tap][c_in][c_out]
        assert torch.equal(kn, want_kn), "pack_kn"
        assert torch.equal(nk, want_nk), "pack_nk"


def test_philox_normal_statistics_and_partition_invariance():
    vf = VF()
    from vae_gan_b200 import _lib
    n = 1 << 20
    full = torch.empty(n, dtype=torch.float32, device=dev())
    _lib.call("vg_philox_normal", full.data_ptr(), n, 77, 5, None, 0, _lib.stream_ptr())
    part = torch.empty(n // 4, dtype=torch.float32, device=dev())
    _lib.call("vg_philox_normal", part.data_ptr(), n // 4, 77, 5, None, n // 2, _lib.stream_ptr())
    assert torch.equal(part, full[n // 2: n // 2 + n // 4])
    assert abs(float(full.mean())) < 5e-3 and abs(float(full.std()) - 1.0) < 5e-3
    assert abs(float((full ** 4).mean()) - 3.0) < 0.05


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c,drop", [(1, 0.5), (6, 0.5), (64, 0.5), (256, 0.0), (10, 0.0)])
def test_bn_act_forward_backward(dtype, c, drop):
    vf = VF()
    tol = TOL32 if dtype == torch.float32 else TOL16
    n, h, w = 4, 12, 12
    xa, _ = rand_act((n, c, h, w), dtype, 1, scale=1.7, shift=0.4)
    gya, _ = rand_act((n, c, h, w), dtype, 2)
    bn = torch.nn.BatchNorm2d(c).to(dev())
    g = torch.Generator().manual_seed(3)
    bn.weight.data = (1 + 0.3 * torch.randn(c, generator=g)).to(dev())
    bn.bias.data = (0.2 * torch.randn(c, generator=g)).to(dev())
    vf.rng.reset_sites()
    xin = xa.detach().clone().requires_grad_(True)
    y = vf.bn_act(xin, bn, slope=0.01, drop_p=drop, training=True)
    y.backward(gya)
    # reference in fp32 on the same (rounded) inputs
    xr = xa.detach().float().clone().requires_grad_(True)
    gam = bn.weight.detach().clone().requires_grad_(True)
    bet = bn.bias.detach().clone().requires_grad_(True)
    yr = F.leaky_relu(F.batch_norm(xr, None, None, gam, bet, True, 0.1, 1e-5), 0.01)
    if drop > 0:
        keep = philox_mask_nchw((n, c, h, w), vf.rng.seed, 0, drop).to(dev())
        yr = yr * keep.float() / (1 - drop)
    yr.backward(gya.float())
    assert_close(y, yr, tol, "y")
    assert_close(xin.grad, xr.grad, tol * (1 if dtype == torch.float32 else 1.5), "dx")
    assert_close(bn.weight.grad, gam.grad, max(tol, 2e-5) if dtype == torch.float32 else tol, "dgamma")
    assert_close(bn.bias.grad, bet.grad, max(tol, 2e-5) if dtype == torch.float32 else tol, "dbeta")
    mean = xa.detach().float().mean((0, 2, 3))
    var = xa.detach().float().var((0, 2, 3), unbiased=True)
    assert_close(bn.running_mean, 0.1 * mean, 1e-5, "running_mean")
    assert_close(bn.running_var, 0.9 + 0.1 * var, 1e-5, "running_var")
    assert int(bn.num_batches_tracked) == 1
    # eval mode uses running statistics
    bn.eval()
    ye = vf.bn_act(xa.detach(), bn, slope=0.01, drop_p=drop, training=False)
    yer = F.leaky_relu(F.batch_norm(xa.detach().float(), bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.1, 1e-5), 0.01)
    assert_close(ye, yer, tol, "eval y")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c,bn_a,bn_b,slope", [(64, False, True, 1.0), (6, True, True, 0.2), (1, False, True, 1.0),
                                               (128, False, False, 1.0), (10, True, False, 0.01)])
def test_bn_add_forward_backward(dtype, c, bn_a, bn_b, slope):
    vf = VF()
    tol = TOL32 if dtype == torch.float32 else TOL16
    n, h, w = 3, 8, 8
    a, _ = rand_act((n, c, h, w), dtype, 5, 1.3, 0.2)
    b, _ = rand_act((n, c, h, w), dtype, 6, 0.7, -0.1)
    gy, _ = rand_act((n, c, h, w), dtype, 7)
    mods = []
    for flag, sd in ((bn_a, 8), (bn_b, 9)):
        if not flag:
            mods.append(None)
            continue
        m = torch.nn.BatchNorm2d(c).to(dev())
        g = torch.Generator().manual_seed(sd)
        m.weight.data = (1 + 0.3 * torch.randn(c, generator=g)).to(dev())
        m.bias.data = (0.2 * torch.randn(c, generator=g)).to(dev())
        mods.append(m)
    ai = a.detach().clone().requires_grad_(True)
    bi = b.detach().clone().requires_grad_(True)
    stats = vf.zeros_f64(2 * c, dev())
    out = vf.bn_add(ai, bi, mods[0], mods[1], slope=slope, training=True, stats_out=stats)
    out.backward(gy)
    ar = a.detach().float().clone().requires_grad_(True)
    br = b.detach().float().clone().requires_grad_(True)
    refp = []
    ta, tb = ar, br
    for i, m in enumerate(mods):
        if m is None:
            refp.append(None)
            continue
        gm = m.weight.detach().clone().requires_grad_(True)
        bt = m.bias.detach().clone().requires_grad_(True)
        refp.append((gm, bt))
        if i == 0:
            ta = F.batch_norm(ar, None, None, gm, bt, True, 0.1, 1e-5)
        else:
            tb = F.batch_norm(br, None, None, gm, bt, True, 0.1, 1e-5)
    outr = F.leaky_relu(ta + tb, slope)
    outr.backward(gy.float())
    assert_close(out, outr, tol, "out")
    assert_close(ai.grad, ar.grad, tol * 1.5, "da")
    assert_close(bi.grad, br.grad, tol * 1.5, "db")
    for m, rp in zip(mods, refp):
        if m is not None:
            assert_close(m.weight.grad, rp[0].grad, max(tol, 3e-5), "dgamma")
            assert_close(m.bias.grad, rp[1].grad, max(tol, 3e-5), "dbeta")
    o32 = out.detach().float()
    assert_close(stats[:c].float(), o32.sum((0, 2, 3)), 1e-5 if dtype == torch.float32 else 1e-4, "stats sum")
    assert_close(stats[c:].float(), (o32 * o32).sum((0, 2, 3)), 1e-5 if dtype == torch.float32 else 1e-4, "stats sumsq")


# ------------------------------------------------------------------------------------------------
CONV_CASES_F32 = [
    # cin, cout, k, stride, pad, transposed, n, h
    (1, 64, 3, 1, 1, False, 2, 12),
    (64, 1, 3, 1, 1, False, 2, 12),
    (1, 1, 3, 1, 1, False, 2, 9),
    (6, 10, 3, 1, 1, False, 3, 8),
    (6, 10, 3, 2, 1, False, 3, 8),
    (6, 10, 4, 2, 1, True, 3, 8),
    (8, 16, 1, 2, 0, False, 2, 8),
    (16, 8, 1, 1, 0, False, 2, 7),
    (16, 24, 3, 1, 1, False, 2, 6),
    (1, 64, 3, 1, 1, False, 2, 16),        # width % 8 == 0: strip kernels
    (64, 1, 3, 1, 1, False, 2, 16),
    (1, 16, 3, 1, 1, False, 3, 8),
]
CONV_CASES_TC = [
    (64, 64, 3, 1, 1, False, 2, 16),
    (64, 128, 3, 1, 1, False, 3, 24),      # 24x24 -> boxes spanning two images, odd batch (padded)
    (128, 128, 3, 1, 1, False, 2, 24),
    (64, 128, 3, 2, 1, False, 2, 16),
    (128, 256, 3, 2, 1, False, 2, 24),
    (128, 64, 4, 2, 1, True, 2, 8),
    (256, 128, 4, 2, 1, True, 3, 12),
    (64, 128, 1, 1, 0, False, 2, 16),
    (128, 256, 1, 2, 0, False, 2, 16),
    (256, 256, 3, 1, 1, False, 1, 12),
    (512, 512, 3, 1, 1, False, 2, 6),
    (64, 1, 3, 1, 1, False, 2, 16),        # single output channel through the tensor-core kernel
    (64, 1, 3, 1, 1, False, 3, 24),
    (64, 128, 3, 1, 1, False, 16, 96),     # enough tiles for the CTA-pair kernel: forward runs pair<128,2,4,8>
    (128, 256, 3, 1, 1, False, 8, 96),     # persistent <256,1,4,8>
    (64, 64, 3, 1, 1, False, 16, 96),      # persistent <64,4,3,4>
]


def _conv_ref(x, w, b, stride, pad, transposed):
    if transposed:
        return F.conv_transpose2d(x, w, b, stride, pad)
    return F.conv2d(x, w, b, stride, pad)


def _run_conv_case(case, dtype, tol, use_bias=False, colscale=False, force_simt=False, out_dtype=None):
    vf = VF()
    from vae_gan_b200 import _lib
    cin, cout, k, stride, pad, transposed, n, h = case
    g = torch.Generator().manual_seed(cin * 131 + cout * 7 + k + stride)
    x = torch.randn(n, cin, h, h, generator=g)
    wshape = (cin, cout, k, k) if transposed else (cout, cin, k, k)
    w = (torch.randn(wshape, generator=g) / math.sqrt(cin * k * k)).to(dev()).requires_grad_(True)
    b = (0.1 * torch.randn(cout, generator=g)).to(dev()).requires_grad_(True) if use_bias else None
    cs = None
    if colscale:
        cs = ((torch.rand(n, cout, generator=g) > 0.5).float() * 2).to(dev())
    xa = vf.as_act(x.to(dev()), dtype).detach().requires_grad_(True)
    prev = _lib.load().vg_set_force_simt(1 if force_simt else 0)
    try:
        geom = vf.ConvGeom(k, stride, pad, transposed)
        stats = vf.zeros_f64(2 * cout, dev())
        y = vf.conv(xa, w, b, geom=geom, colscale=cs, stats_out=stats, out_dtype=out_dtype)
        gy = torch.randn(y.shape, generator=g).to(dev())
        gya = vf.as_act(vf.as_act(gy, dtype), y.dtype)      # dtype-rounded values, in y's dtype
        y.backward(gya)
    finally:
        _lib.load().vg_set_force_simt(prev)
    # reference: fp32 math on the rounded operands
    xr = xa.detach().float().clone().requires_grad_(True)
    wq = w.detach().to(dtype).float().requires_grad_(True)
    br = b.detach().clone().requires_grad_(True) if use_bias else None
    yr = _conv_ref(xr, wq, br, stride, pad, transposed)
    if cs is not None:
        yr = yr * cs[:, :, None, None]
    yr.backward(gya.float() if cs is None else gya.float())
    # NOTE: with colscale the product's ConvFn expects the UNSCALED-output gradient (its partner
    # BnActFn applies the scale); so for the gradient comparison feed the reference accordingly
    if cs is not None:
        xr.grad = None
        wq.grad = None
        y2 = _conv_ref(xr, wq, None, stride, pad, transposed)
        y2.backward(gya.float())
    e = {}
    e["y"] = assert_close(y, yr, tol, f"{case} y")
    e["dx"] = assert_close(xa.grad, xr.grad, tol, f"{case} dx")
    e["dw"] = assert_close(w.grad, wq.grad, tol, f"{case} dw")
    if use_bias:
        e["db"] = assert_close(b.grad, br.grad, tol, f"{case} db")
    yv = y.detach().float()
    assert_close(stats[:cout].float(), yv.sum((0, 2, 3)), 1e-4, "stats sum")
    assert_close(stats[cout:].float(), (yv * yv).sum((0, 2, 3)), 1e-4, "stats sumsq")
    return e


@pytest.mark.parametrize("case", CONV_CASES_F32)
def test_conv_fp32_simt(case):
    _run_conv_case(case, torch.float32, TOL32 * 2, use_bias=(case[0] == 16), colscale=(case[1] == 10 and not case[5]))


@pytest.mark.parametrize("case", CONV_CASES_F32 + CONV_CASES_TC[:3])
def test_conv_bf16_simt(case):
    _run_conv_case(case, torch.bfloat16, TOL16, force_simt=True)


@pytest.mark.parametrize("case", CONV_CASES_TC)
def test_conv_bf16_tensor_core(case):
    e = _run_conv_case(case, torch.bfloat16, TOL16)
    # the tensor-core result is fp32-accumulated: far tighter than the bf16 storage tolerance
    assert e["dw"] < 2e-3, e


def test_conv_tensor_core_bias_colscale_fp32_out():
    _run_conv_case((256, 256, 3, 1, 1, False, 2, 12), torch.bfloat16, TOL16, use_bias=True, out_dtype=torch.float32)
    _run_conv_case((64, 128, 3, 2, 1, False, 4, 16), torch.bfloat16, TOL16, colscale=True)


def test_tensor_core_matches_simt_bitwise_inputs():
    """Same bf16 inputs through the tcgen05 kernel and the CUDA-core kernel: both accumulate in
    fp32, so they agree to accumulation-order noise (a check that needs no external reference)."""
    vf = VF()
    from vae_gan_b200 import _lib
    g = torch.Generator().manual_seed(5)
    x = vf.as_act(torch.randn(2, 128, 24, 24, generator=g).to(dev()), torch.bfloat16)
    w = (torch.randn(128, 128, 3, 3, generator=g) / 34.0).to(dev())
    geom = vf.ConvGeom(3, 1, 1, False)
    y_tc = vf.conv(x, w, None, geom=geom, out_dtype=torch.float32)
    prev = _lib.load().vg_set_force_simt(1)
    try:
        y_simt = vf.conv(x, w, None, geom=geom, out_dtype=torch.float32)
    finally:
        _lib.load().vg_set_force_simt(prev)
    assert_close(y_tc, y_simt, 2e-5, "tc vs simt")


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("wdtype", [torch.float32, torch.bfloat16])
def test_linear_forward_backward(wdtype):
    vf = VF()
    tol = 2e-5 if wdtype == torch.float32 else TOL16
    g = torch.Generator().manual_seed(1)
    for m, k, n, slope in [(4, 1152, 64, 0.2), (5, 70, 33, 1.0), (3, 256, 1, 1.0)]:
        x = torch.randn(m, k, generator=g).to(dev()).requires_grad_(True)
        w = (torch.randn(n, k, generator=g) / math.sqrt(k)).to(dev()).requires_grad_(True)
        b = (0.1 * torch.randn(n, generator=g)).to(dev()).requires_grad_(True)
        y = vf.LinearFn.apply(x, w, b, slope, wdtype)
        gy = torch.randn(m, n, generator=g).to(dev())
        y.backward(gy)
        xr = x.detach().clone().requires_grad_(True)
        wr = w.detach().to(wdtype).float().requires_grad_(True)
        br = b.detach().clone().requires_grad_(True)
        yr = F.leaky_relu(F.linear(xr, wr, br), slope)
        yr.backward(gy)
        assert_close(y, yr, tol, "y")
        assert_close(x.grad, xr.grad, tol, "dx")
        assert_close(w.grad, wr.grad, tol, "dw")
        assert_close(b.grad, br.grad, tol, "db")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_avgpool_flatten(dtype):
    vf = VF()
    xa, _ = rand_act((3, 16, 8, 8), dtype, 4)
    xi = xa.detach().clone().requires_grad_(True)
    y = vf.AvgPoolFlattenFn.apply(xi, 4)
    g = torch.randn(y.shape, generator=torch.Generator().manual_seed(1)).to(dev())
    y.backward(g)
    xr = xa.detach().float().clone().requires_grad_(True)
    yr = F.avg_pool2d(xr, 4).reshape(3, -1)
    yr.backward(g)
    assert_close(y, yr, 1e-6, "pool")
    assert_close(xi.grad, xr.grad, 1e-6 if dtype == torch.float32 else 4e-3, "dpool")


def test_spectral_norm_sigma_and_backward():
    vf = VF()
    from vae_gan_b200 import _lib
    g = torch.Generator().manual_seed(2)
    for rows, cols in [(16, 54), (128, 1152), (512, 4608)]:
        w = torch.randn(rows, cols, generator=g) / math.sqrt(cols)
        u = F.normalize(torch.randn(rows, generator=g), dim=0)
        v = F.normalize(torch.randn(cols, generator=g), dim=0)
        P = {"c.weight_orig": w.clone().requires_grad_(True), "c.weight_u": u.clone(), "c.weight_v": v.clone()}
        wn = O.spectral_normed_weight(P, "c", True)
        dwh = torch.randn(rows, cols, generator=g)
        wn.backward(dwh)
        wd, ud, vd = w.to(dev()), u.to(dev()), v.to(dev())
        sigma = torch.empty(1, device=dev())
        ws = torch.empty(rows + cols + 4, device=dev())
        _lib.call("vg_spectral_norm_sigma", wd.data_ptr(), rows, cols, ud.data_ptr(), vd.data_ptr(), 1, 1e-12,
                  sigma.data_ptr(), ws.data_ptr(), _lib.stream_ptr())
        assert_close(ud, P["c.weight_u"], 2e-5, "u")
        assert_close(vd, P["c.weight_v"], 2e-5, "v")
        sig_ref = (P["c.weight_orig"].detach() / wn.detach())[0, 0]
        assert abs(float(sigma) - float(sig_ref)) <= 2e-5 * abs(float(sig_ref))
        dw = torch.zeros(rows, cols, device=dev())
        _lib.call("vg_spectral_norm_backward", dwh.to(dev()).data_ptr(), wd.data_ptr(), ud.data_ptr(), vd.data_ptr(),
                  sigma.data_ptr(), rows, cols, dw.data_ptr(), ws.data_ptr(), _lib.stream_ptr())
        assert_close(dw, P["c.weight_orig"].grad, 3e-5, "dw_orig")
        # eval: no update, sigma from the stored u, v
        u2, v2 = ud.clone(), vd.clone()
        _lib.call("vg_spectral_norm_sigma", wd.data_ptr(), rows, cols, u2.data_ptr(), v2.data_ptr(), 0, 1e-12,
                  sigma.data_ptr(), ws.data_ptr(), _lib.stream_ptr())
        assert torch.equal(u2, ud) and torch.equal(v2, vd)
        Pe = {"c.weight_orig": w, "c.weight_u": ud.cpu(), "c.weight_v": vd.cpu()}
        sig_e = (w / O.spectral_normed_weight(Pe, "c", False))[0, 0]
        assert abs(float(sigma) - float(sig_e)) <= 2e-5 * abs(float(sig_e))


def test_reparam_and_losses_match_oracle():
    vf = VF()
    g = torch.Generator().manual_seed(9)
    n, c, h = 3, 16, 6
    mu = torch.randn(n, c, h, h, generator=g)
    lv_raw = torch.randn(n, c, h, h, generator=g) * 30          # exercises the +-50 clamp
    eps = torch.randn(n, c, h, h, generator=g)
    xhat = torch.randn(n, 1, 24, 24, generator=g)
    x = torch.rand(n, 1, 24, 24, generator=g)
    logits = torch.randn(n, 1, generator=g)
    for adv_mode, name in ((0, "bce"), (1, "wgan")):
        mu_r = mu.clone().requires_grad_(True)
        lv_r = lv_raw.clone().requires_grad_(True)
        xh_r = xhat.clone().requires_grad_(True)
        lg_r = logits.clone().requires_grad_(True)
        lvc = torch.clamp(lv_r, -50, 50)
        z_r = mu_r + torch.exp(0.5 * lvc) * eps
        total_r = 1.0 * O.g_adv_loss(lg_r, name) + 10.0 * O.reconstruction_loss(xh_r, x) + 0.1 * O.kl_divergence(mu_r, lvc)
        gz = torch.randn(z_r.shape, generator=g) * 1e-3
        (total_r + (z_r * gz).sum()).backward()

        mu_d = vf.as_act(mu.to(dev()), torch.float32).requires_grad_(True)
        lv_d = vf.as_act(lv_raw.to(dev()), torch.float32).requires_grad_(True)
        xh_d = vf.as_act(xhat.to(dev()), torch.float32).requires_grad_(True)
        lg_d = logits.to(dev()).requires_grad_(True)
        z, lv = vf.ReparamFn.apply(mu_d, lv_d, vf.as_act(eps.to(dev()), torch.float32), True, torch.float32)
        tot, recon, kl, adv = vf.GeneratorLossFn.apply(xh_d, x.to(dev()), mu_d, lv, lg_d, adv_mode, 1.0, 10.0, 0.1)
        (tot + (z * vf.as_act(gz.to(dev()), torch.float32)).sum()).backward()
        assert_close(z, z_r, 1e-5, "z")
        assert abs(float(tot) - float(total_r)) <= 1e-5 * abs(float(total_r))
        assert abs(float(kl) - float(O.kl_divergence(mu, torch.clamp(lv_raw, -50, 50)))) <= 1e-5 * abs(float(kl))
        assert_close(mu_d.grad, mu_r.grad, 1e-5, "dmu")
        assert_close(lv_d.grad, lv_r.grad, 1e-5, "dlv")
        assert_close(xh_d.grad, xh_r.grad, 1e-5, "dxhat")
        assert_close(lg_d.grad, lg_r.grad, 1e-5, "dlogits")
        # discriminator loss
        dr = torch.randn(n, 1, generator=g)
        df = torch.randn(n, 1, generator=g)
        dr_r, df_r = dr.clone().requires_grad_(True), df.clone().requires_grad_(True)
        a, b = O.d_loss_terms(dr_r, df_r, name)
        (a + b).backward()
        dr_d, df_d = dr.to(dev()).requires_grad_(True), df.to(dev()).requires_grad_(True)
        t, lr_, lf_ = vf.DiscriminatorLossFn.apply(dr_d, df_d, adv_mode)
        t.backward()
        assert abs(float(t) - float(a + b)) <= 1e-5 * max(1.0, abs(float(a + b)))
        assert_close(dr_d.grad, dr_r.grad, 1e-5, "d_real grad")
        assert_close(df_d.grad, df_r.grad, 1e-5, "d_fake grad")


@pytest.mark.parametrize("kind", ["adam", "rmsprop"])
def test_fused_optimizer_matches_oracle(kind):
    vf = VF()
    g = torch.Generator().manual_seed(4)
    n = 10007
    p0 = torch.randn(n, generator=g)
    P = {"w": p0.clone()}
    st = O.OptState(kind=kind, lr=3e-4, weight_decay=0.0 if kind == "adam" else 1e-5)
    p = p0.to(dev())
    m = torch.zeros(n, device=dev())
    v = torch.zeros(n, device=dev())
    step_t = torch.zeros(1, dtype=torch.int64, device=dev())
    for it in range(1, 6):
        gr = torch.randn(n, generator=g)
        O.optimizer_step(P, {"w": gr}, st)
        step_t += 1
        vf.optimizer_step(p, gr.to(dev()), m, v, kind=kind, lr=3e-4, weight_decay=st.weight_decay,
                          step_tensor=step_t if it % 2 else None, step=it)
    assert_close(p, P["w"], 2e-6, "params")
    # clamp (README.md:805-806)
    vf.optimizer_step(p, torch.zeros(n, device=dev()), m, v, kind=kind, lr=0.0, clamp=0.01, step=6)
    assert float(p.abs().max()) <= 0.01 + 1e-9


def test_layout_helpers_roundtrip():
    vf = VF()
    from vae_gan_b200 import _lib
    x = torch.randn(3, 10, 7, 5, generator=torch.Generator().manual_seed(0)).to(dev())
    for dt in (torch.float32, torch.bfloat16):
        a = vf.as_act(x, dt)
        assert vf.is_act(a) and a.shape == x.shape
        assert_close(a, x.to(dt).float(), 1e-7, "nchw->nhwc")
        back = torch.empty_like(x)
        _lib.call("vg_nhwc_to_nchw", a.data_ptr(), _lib.vg_dtype(dt), 3, 10, 7, 5, back.data_ptr(), _lib.stream_ptr())
        assert_close(back, x.to(dt).float(), 1e-7, "nhwc->nchw")


def test_unsupported_and_invalid_arguments_raise():
    vf = VF()
    from vae_gan_b200 import _lib
    with pytest.raises(_lib.VgError):
        _lib.call("vg_bn_stats", None, None, None, _lib.stream_ptr())
    d = _lib.VgConvDesc(1, 8, 8, 4, 9, 9, 4, 3, 3, 1, 1, 0, 0, 0)   # inconsistent output dims
    with pytest.raises(_lib.VgError):
        _lib.call("vg_conv_forward", C.byref(d), 1, 1, 1, None, None, 1, None, _lib.stream_ptr())
    # empty batch is a no-op, not an error
    x = vf.empty_act(0, 8, 4, 4, torch.float32, dev())
    w = torch.randn(8, 8, 3, 3, device=dev())
    y = vf.conv(x, w, None, geom=vf.ConvGeom(3, 1, 1, False))
    assert y.shape == (0, 8, 4, 4)
