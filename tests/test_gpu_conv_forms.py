"""Every tensor-core convolution kernel form and epilogue against an fp64 reference, element by element (-m gpu).

The kernels are called through the C ABI (vg_conv_forward_fused, vg_conv_dgrad_scaled, vg_conv_wgrad) on bf16 NHWC tensors.
The reference computes the same operation in float64 with plain torch on exactly the operands the kernel sees (the bf16
activations and bf16-representable weights, so the weight pack is exact).  Next to it the same operation on absolute values,
A = conv(|x|, |W|) (with |sigma|, |bias| and |colscale| applied as in the epilogue), bounds the fp32 accumulation error of
each output element: acc = 8 sqrt(K) 2^-24 A, K = taps x reduction channels (pixels for the weight gradient).

  - fp32 outputs: |got - ref| <= acc + ulp32(ref) per element, and the max-normalised error is <= 1e-5;
  - bf16 outputs: |got - ref| <= ulp_bf16(ref) + acc per element, and >= 99 % of the elements are within half an ulp plus
    acc - a kernel that truncates instead of rounding to nearest passes the first clause but not the second.

The kernel form (one-shot CTAs, persistent CTAs, CTA pairs) and the N tile are pinned per case through the tile table
(vae_gan_b200/tune.py); a form the shape cannot take falls back to the next one, so the cases are chosen to make each
kernel instance run: test_every_tensor_core_kernel_instance_runs checks that with the profiler.
"""
import ctypes as C
import math
import re
import zlib
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

ACC_FACTOR = 8.0
VG_EUNSUPPORTED = -4


# ---- error bound (CPU-testable) ----------------------------------------------------------------------------------------
def ulp_bf16(ref: torch.Tensor) -> torch.Tensor:
    """Spacing of bf16 numbers (8 significant bits) at |ref|, float64; subnormal spacing below the smallest normal."""
    ref = ref.double()
    _, e = torch.frexp(ref)                       # |ref| = m 2^e, m in [0.5, 1)
    u = torch.ldexp(torch.ones_like(ref), e - 8)
    return torch.where(ref.abs() < 2.0 ** -126, torch.full_like(ref, 2.0 ** -133), u)


def ulp_f32(ref: torch.Tensor) -> torch.Tensor:
    ref = ref.double()
    _, e = torch.frexp(ref)
    u = torch.ldexp(torch.ones_like(ref), e - 24)
    return torch.where(ref.abs() < 2.0 ** -126, torch.full_like(ref, 2.0 ** -149), u)


def acc_bound(A: torch.Tensor, K: int) -> torch.Tensor:
    """Accumulation allowance of an fp32 sum of K products whose absolute values sum to A."""
    return ACC_FACTOR * math.sqrt(K) * 2.0 ** -24 * A.double()


def check_bound(got, ref, acc, name, half_ulp_frac=0.99):
    """The per-element bound of the module docstring for got's dtype (bf16 or fp32).  Returns the largest |got - ref| / acc
    (the measurement behind ACC_FACTOR; for bf16 outputs the rounding to bf16 dominates it)."""
    g = got.double()
    ref = ref.double().to(g.device)
    acc = acc.double().to(g.device)
    err = (g - ref).abs()
    assert torch.isfinite(g).all(), f"{name}: non-finite output"
    if got.dtype == torch.bfloat16:
        u = ulp_bf16(ref)
        bad = err > u + acc
        assert not bad.any(), (f"{name}: {int(bad.sum())} of {bad.numel()} elements off by more than one bf16 ulp + acc; "
                               f"worst {float((err - u - acc).max()):.3e} at {_where(bad)}")
        frac = float((err <= 0.5 * u + acc).double().mean())
        assert frac >= half_ulp_frac, f"{name}: only {100 * frac:.2f} % of elements within half a bf16 ulp + acc (rounding bias?)"
    else:
        assert got.dtype == torch.float32, got.dtype
        bad = err > acc + ulp_f32(ref)
        assert not bad.any(), (f"{name}: {int(bad.sum())} of {bad.numel()} elements off by more than acc + one fp32 ulp; "
                               f"worst {float((err - acc - ulp_f32(ref)).max()):.3e} at {_where(bad)}")
        rel = float(err.max()) / max(float(ref.abs().max()), 1e-300)
        assert rel <= 1e-5, f"{name}: max-normalised error {rel:.3e} > 1e-5"
    nz = acc > 0
    return float((err[nz] / acc[nz]).max()) if bool(nz.any()) else 0.0


def _where(mask):
    idx = mask.nonzero()
    return tuple(idx[0].tolist()) if len(idx) else None


def test_bound_helper_accepts_round_to_nearest_and_rejects_truncation():
    g = torch.Generator().manual_seed(0)
    ref = (torch.randn(4096, generator=g, dtype=torch.float64) * torch.exp(4 * torch.randn(4096, generator=g, dtype=torch.float64)))
    zero = torch.zeros_like(ref)
    rn = ref.float().to(torch.bfloat16)                                               # float32 -> bf16 rounds to nearest
    check_bound(rn, ref, zero, "round to nearest")
    trunc = (ref.float().view(torch.int32) & -65536).view(torch.float32).to(torch.bfloat16)   # drop the low 16 bits
    assert torch.equal(trunc.float().view(torch.int32) & 0xFFFF, torch.zeros(4096, dtype=torch.int32))
    with pytest.raises(AssertionError, match="rounding bias"):
        check_bound(trunc, ref, zero, "truncated")
    two_ulp = (rn.double() + 2 * ulp_bf16(rn.double())).to(torch.bfloat16)           # two ulps off: the per-element clause
    with pytest.raises(AssertionError, match="more than one bf16 ulp"):
        check_bound(two_ulp, ref, zero, "two ulps")
    # the accumulation allowance widens the bound (two ulps of rn are up to four of ref where rn rounded up to a power of 2)
    check_bound(two_ulp, ref, 4 * ulp_bf16(ref), "two ulps within acc")
    # fp32: round to nearest passes, an error of a few ulps does not
    check_bound(ref.float(), ref, zero, "fp32 round to nearest")
    with pytest.raises(AssertionError, match="fp32 ulp"):
        check_bound((ref + 4 * ulp_f32(ref)).float(), ref, zero, "fp32 four ulps")
    assert float(ulp_bf16(torch.tensor([1.0, 1.5, -3.0, 2.0 ** -130]).double()).sub(
        torch.tensor([2.0 ** -7, 2.0 ** -7, 2.0 ** -6, 2.0 ** -133]).double()).abs().max()) == 0.0


# ---- cases -------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class Case:
    n: int
    cin: int
    cout: int
    h: int
    w: int
    k: int
    st: int
    pad: int
    tr: int = 0

    @property
    def out_hw(self):
        if self.tr:
            return (self.h - 1) * self.st - 2 * self.pad + self.k, (self.w - 1) * self.st - 2 * self.pad + self.k
        return (self.h + 2 * self.pad - self.k) // self.st + 1, (self.w + 2 * self.pad - self.k) // self.st + 1

    def key(self, dgrad):
        return (int(dgrad), self.n, self.h, self.w, self.cin, self.cout, self.k, self.st, self.pad, self.tr)

    def wshape(self):
        return (self.cin, self.cout, self.k, self.k) if self.tr else (self.cout, self.cin, self.k, self.k)


def _cdiv(a, b):
    return -(-a // b)


def _choose_box(gw, gh, gn, pixels=128):
    """tc_conv_run's choose_box: the {TW, TH, TN} box of 128 GEMM rows with the least padded work."""
    best, bw, bh = 1e30, 1, 1
    tw = 1
    while tw <= pixels:
        th = 1
        while tw * th <= pixels:
            tn = pixels // (tw * th)
            if tw <= 256 and th <= 256 and tn <= 256:
                score = _cdiv(gw, tw) * tw * _cdiv(gh, th) * th * _cdiv(gn, tn) * tn - 1e-3 * tw - 1e-6 * th
                if score < best:
                    best, bw, bh = score, tw, th
            th *= 2
        tw *= 2
    return bw, bh, pixels // (bw * bh)


def pixel_tiles(c: Case, dgrad: bool) -> int:
    """Number of 128-pixel tiles tc_conv_run launches per phase (grid.x): the count the persistent kernels group by MT
    and the pair kernels need divisible by 2 MT (MT = 4 / 2 / 1 for 64 / 128 / 256-wide tiles)."""
    ho, wo = c.out_hw
    gather = bool(c.tr) == dgrad
    oh, ow = (c.h, c.w) if dgrad else (ho, wo)
    gw, gh = (ow, oh) if gather else (_cdiv(ow, c.st), _cdiv(oh, c.st))
    tw, th, tn = _choose_box(gw, gh, c.n)
    return _cdiv(gw, tw) * _cdiv(gh, th) * _cdiv(c.n, tn)


MT = {64: 4, 128: 2, 256: 1}

# Form matrix: forward and dgrad of each case under the heuristic and every (N tile, form) the tile table accepts.
FORM_CASES = {
    # stride-1 gather, non-square 20x12 (ragged 16x8 boxes), odd batch; 9 tiles: a last persistent group of fewer than MT
    "s1_20x12": Case(3, 64, 128, 20, 12, 3, 1, 1),
    # stride-2 gather through the parity maps, non-square; dgrad = 4 scatter phases.  2 tiles: pair<256> runs, pair<64/128>
    # fall back to the persistent kernel
    "s2_24x16": Case(2, 128, 256, 24, 16, 3, 2, 1),
    "s2_32x16": Case(4, 256, 256, 32, 16, 3, 2, 1),          # 4 tiles: pair<128> and pair<256> run, pair<64> falls back
    # ConvTranspose2d 4x4 stride 2: 4 scatter phases of 4 taps each (12x8 -> 24x16); dgrad = stride-2 gather
    "tr_12x8": Case(3, 256, 128, 12, 8, 4, 2, 1, 1),
    "tr_16x8": Case(8, 256, 128, 16, 8, 4, 2, 1, 1),          # 8 tiles: every pair form runs, scatter and gather
    # 1x1 stride 2: dgrad has three phases without taps (zero outputs)
    "1x1_s2": Case(2, 128, 256, 16, 24, 1, 2, 0),
    # 1x1 stride 1, one k-block (c_red = 64) both ways; 24x24 boxes span images, odd batch
    "1x1_s1": Case(3, 64, 64, 24, 24, 1, 1, 0),
    # long ring: c_red = 1024 at 3x3 = 144 k-blocks (forward)
    "ring_1024": Case(2, 1024, 128, 8, 12, 3, 1, 1),
    # 2592 tiles: at least four work items per persistent CTA / CTA pair (the TMEM double buffer wraps its parity)
    "64_96x96_b36": Case(36, 64, 64, 96, 96, 3, 1, 1),
    # single output channel: 64->1 forward, 1->64 dgrad (no pair form: falls back to the persistent kernel)
    "out1_20x12": Case(3, 64, 1, 20, 12, 3, 1, 1),
    "in1_20x12": Case(3, 1, 64, 20, 12, 3, 1, 1),
}
# the epilogue case: 64->256 at 16x32 (32x4 boxes), batch 6: 24 tiles, so all three forms run with all three N tiles
EP = Case(6, 64, 256, 16, 32, 3, 1, 1)


def test_case_table_reaches_every_tile_count_class():
    """The cases above make each kernel instance's tile-count condition happen (the profiler test checks the launches)."""
    counts = {(nm, dg): pixel_tiles(c, dg) for nm, c in list(FORM_CASES.items()) + [("EP", EP)] for dg in (False, True)}
    for bn, mt in MT.items():
        assert any(t % (2 * mt) == 0 for t in counts.values()), f"no case runs pair<{bn}>"
        assert any(t % (2 * mt) != 0 and t > 0 for t in counts.values()), f"no case falls back from pair<{bn}>"
        assert any(t % mt != 0 for t in counts.values()) or mt == 1, f"no ragged last group for MT={mt}"
    assert pixel_tiles(EP, False) % 8 == 0
    assert pixel_tiles(FORM_CASES["64_96x96_b36"], False) // 8 >= 4 * 74       # >= 4 items per CTA pair (148 SMs)
    assert pixel_tiles(FORM_CASES["64_96x96_b36"], False) // 4 >= 4 * 148       
    assert _choose_box(32, 16, 6) == (32, 4, 1)                                  # TW != TH: a swapped origin shows


# ---- GPU plumbing ------------------------------------------------------------------------------------------------------
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    import vae_gan_b200  # noqa: F401
    from vae_gan_b200 import _lib
    _lib.ensure_device(dev())
    return _lib


def _desc(c: Case, out_dtype=torch.bfloat16, act_dtype=torch.bfloat16):
    from vae_gan_b200 import _lib
    ho, wo = c.out_hw
    return _lib.VgConvDesc(c.n, c.h, c.w, c.cin, ho, wo, c.cout, c.k, c.k, c.st, c.pad, c.tr,
                           _lib.vg_dtype(act_dtype), _lib.vg_dtype(out_dtype))


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _nchw(t):
    return t.permute(0, 3, 1, 2)


class Operands:
    """Seeded bf16 operands of one case (NHWC on the device) and their fp64 NCHW copies; the weight is bf16-representable
    fp32 in torch layout, packed by the library."""

    def __init__(self, c: Case, seed, act_dtype=torch.bfloat16):
        from vae_gan_b200 import _lib
        g = torch.Generator(device=dev()).manual_seed(seed)
        ho, wo = c.out_hw
        self.c = c
        self.x = torch.randn(c.n, c.h, c.w, c.cin, generator=g, device=dev()).to(act_dtype)
        self.dy = torch.randn(c.n, ho, wo, c.cout, generator=g, device=dev()).to(act_dtype)
        fan = c.cin * c.k * c.k if not c.tr else c.cout * c.k * c.k
        self.w = (torch.randn(c.wshape(), generator=g, device=dev()) / math.sqrt(fan)).to(act_dtype).float()
        d = _desc(c, act_dtype=act_dtype, out_dtype=act_dtype)
        self.pk = torch.empty(self.w.numel(), dtype=act_dtype, device=dev())
        self.pn = torch.empty_like(self.pk)
        _lib.call("vg_conv_pack_weights", C.byref(d), self.w.data_ptr(), None, self.pk.data_ptr(), self.pn.data_ptr(),
                  _lib.stream_ptr())
        self.x64, self.dy64, self.w64 = _nchw(self.x).double(), _nchw(self.dy).double(), self.w.double()


def fwd64(c: Case, x, w):
    if c.tr:
        return F.conv_transpose2d(x, w, stride=c.st, padding=c.pad)
    return F.conv2d(x, w, stride=c.st, padding=c.pad)


def dgrad64(c: Case, dy, w):
    if c.tr:
        return F.conv2d(dy, w, stride=c.st, padding=c.pad)
    return torch.nn.grad.conv2d_input((c.n, c.cin, c.h, c.w), w, dy, stride=c.st, padding=c.pad)


def wgrad64(c: Case, x, dy):
    if c.tr:
        return torch.nn.grad.conv2d_weight(dy, c.wshape(), x, stride=c.st, padding=c.pad)
    return torch.nn.grad.conv2d_weight(x, c.wshape(), dy, stride=c.st, padding=c.pad)


def k_len(c: Case, dgrad: bool) -> int:
    """Reduction length of one output element: taps x reduction channels (for the scatter phases an upper bound)."""
    return c.k * c.k * (c.cout if dgrad else c.cin)


def run_forward(lib, ops: Operands, out_dtype=torch.bfloat16, bias=None, colscale=None, sigma=None, sigma_group_n=0,
                act_slope=1.0, residual=None, y2=False, post=None, raw=False):
    c = ops.c
    ho, wo = c.out_hw
    y = torch.full((c.n, ho, wo, c.cout), float("nan"), dtype=out_dtype, device=dev())
    y2t = torch.full_like(y, float("nan")) if y2 else None
    ps, pt, pslope = post if post is not None else (None, None, 1.0)
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    ep = lib.VgConvEpilogue(ptr(bias), ptr(colscale), ptr(sigma), sigma_group_n, act_slope, ptr(residual), ptr(y2t),
                            ptr(ps), ptr(pt), pslope)
    d = _desc(c, out_dtype, ops.x.dtype)
    args = (C.byref(d), ops.x.data_ptr(), ops.pk.data_ptr(), ops.pn.data_ptr(), C.byref(ep), y.data_ptr(), None, lib.stream_ptr())
    if raw:
        return lib.load().vg_conv_forward_fused(*args)
    lib.call("vg_conv_forward_fused", *args)
    return (y, y2t) if y2 else y


def run_dgrad(lib, ops: Operands, sigma=None, sigma_group_n=0):
    c = ops.c
    dx = torch.full((c.n, c.h, c.w, c.cin), float("nan"), dtype=ops.x.dtype, device=dev())
    d = _desc(c, ops.x.dtype, ops.x.dtype)
    lib.call("vg_conv_dgrad_scaled", C.byref(d), ops.dy.data_ptr(), ops.pk.data_ptr(), ops.pn.data_ptr(),
             None if sigma is None else sigma.data_ptr(), sigma_group_n, dx.data_ptr(), lib.stream_ptr())
    return dx


def form_configs(n_out):
    """(N tile, form) pairs to pin: (0, 0) = the heuristic (no entry); N tiles that divide n_out (bn 0 keeps the
    heuristic's tile, the only choice for a single output channel) with forms 1 one-shot, 2 persistent, 3 pair."""
    cfgs = [(0, 0)]
    tiles = [bn for bn in (64, 128, 256) if n_out % bn == 0] or [0]
    return cfgs + [(bn, f) for bn in tiles for f in (1, 2, 3)]


def with_forms(c: Case, dgrad: bool, fn):
    """Run fn(cfg) under every form configuration of (c, dgrad); entries are removed afterwards (the shipped table keeps
    its own entries: these shapes are not in it)."""
    from vae_gan_b200 import tune
    key = c.key(dgrad)
    for cfg in form_configs(c.cin if dgrad else c.cout):
        try:
            if cfg != (0, 0):
                tune.set_entry(key, *cfg)
            fn(cfg)
        finally:
            tune.set_entry(key, 0, 0)


def _sgn(group_n, n, sigma):
    """per-sample sigma of a sigma_group_n grouping, shaped for NCHW broadcasting"""
    idx = torch.arange(n, device=sigma.device) // group_n if group_n > 0 else torch.zeros(n, dtype=torch.long, device=sigma.device)
    return sigma.double()[idx].view(n, 1, 1, 1)


def _seed(name):
    return zlib.crc32(name.encode()) % 1000


def _report(tag, ratio):
    print(f"[acc] {tag}: max |got-ref|/acc = {ratio:.3f}")


# ---- 2. kernel-form matrix ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FORM_CASES))
def test_forward_and_dgrad_every_form_vs_fp64(lib, name):
    c = FORM_CASES[name]
    ops = Operands(c, seed=_seed(name))
    for dgrad in (False, True):
        red = c.cout if dgrad else c.cin
        n_out = c.cin if dgrad else c.cout
        if red % 64 != 0 or (n_out % 64 != 0 and n_out != 1):
            continue                                    # not a tensor-core shape in this direction (CUDA-core tests below)
        if dgrad:
            ref, A = dgrad64(c, ops.dy64, ops.w64), dgrad64(c, ops.dy64.abs(), ops.w64.abs())
        else:
            ref, A = fwd64(c, ops.x64, ops.w64), fwd64(c, ops.x64.abs(), ops.w64.abs())
        acc = acc_bound(A, k_len(c, dgrad))

        def one(cfg):
            got = run_dgrad(lib, ops) if dgrad else run_forward(lib, ops)
            r = check_bound(_nchw(got), ref, acc, f"{name} {'dgrad' if dgrad else 'forward'} {cfg}")
            _report(f"{name} {'dgrad' if dgrad else 'fwd'} {cfg} bf16", r)
        with_forms(c, dgrad, one)
    if name == "ring_1024":
        # fp32 output of a long reduction on two tiles: the split-K one-shot kernel (vector atomics into a zeroed output)
        ref, A = fwd64(c, ops.x64, ops.w64), fwd64(c, ops.x64.abs(), ops.w64.abs())
        got = run_forward(lib, ops, out_dtype=torch.float32)
        _report(f"{name} fwd split-K fp32", check_bound(_nchw(got), ref, acc_bound(A, k_len(c, False)), f"{name} fp32 split-K"))


# ---- 3. epilogue matrix ------------------------------------------------------------------------------------------------
def _ep_operands():
    g = torch.Generator(device=dev()).manual_seed(11)
    c = EP
    return dict(
        bias=0.5 * torch.randn(c.cout, generator=g, device=dev()),
        drop=(torch.rand(c.n, c.cout, generator=g, device=dev()) > 0.5).float() * 2.0,     # Dropout2d keep / (1 - p)
        cs=torch.randn(c.n, c.cout, generator=g, device=dev()),
        sigma=torch.tensor([1.7, 0.6, 2.9], device=dev()),
    )


EP_FWD = [
    # name, out dtype, use bias, colscale key, sigma_group_n (None = no sigma)
    ("plain_f32", torch.float32, False, None, None),
    ("bias", torch.bfloat16, True, None, None),
    ("bias_f32", torch.float32, True, None, None),
    ("dropout2d", torch.bfloat16, True, "drop", None),
    ("colscale", torch.bfloat16, False, "cs", None),
    ("colscale_f32", torch.float32, True, "cs", 0),
    ("sigma", torch.bfloat16, False, None, 0),
    ("sigma_groups3", torch.bfloat16, True, "cs", 2),          # samples {0,1} {2,3} {4,5}
    ("sigma_groups2", torch.bfloat16, False, None, 4),         # samples {0..3} {4,5}
    ("sigma_groups3_f32", torch.float32, False, "drop", 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [v[0] for v in EP_FWD])
def test_forward_epilogue_every_form_vs_fp64(lib, variant):
    _, out_dtype, use_bias, cs_key, sgn = next(v for v in EP_FWD if v[0] == variant)
    c = EP
    ops = Operands(c, seed=5)
    e = _ep_operands()
    bias = e["bias"] if use_bias else None
    cs = e[cs_key] if cs_key else None
    sigma = e["sigma"] if sgn is not None else None
    ref, A = fwd64(c, ops.x64, ops.w64), fwd64(c, ops.x64.abs(), ops.w64.abs())
    if sigma is not None:
        s = _sgn(sgn, c.n, sigma)
        ref, A = ref / s, A / s.abs()
    if bias is not None:
        ref, A = ref + bias.double().view(1, -1, 1, 1), A + bias.double().abs().view(1, -1, 1, 1)
    if cs is not None:
        ref, A = ref * cs.double()[:, :, None, None], A * cs.double().abs()[:, :, None, None]
    acc = acc_bound(A, k_len(c, False))

    def one(cfg):
        got = run_forward(lib, ops, out_dtype, bias=bias, colscale=cs, sigma=sigma, sigma_group_n=sgn or 0)
        _report(f"EP fwd {variant} {cfg}", check_bound(_nchw(got), ref, acc, f"forward {variant} {cfg}"))
    with_forms(c, False, one)


@pytest.mark.gpu
@pytest.mark.parametrize("sgn", [0, 2, 4])
def test_dgrad_sigma_every_form_vs_fp64(lib, sgn):
    c = EP
    ops = Operands(c, seed=6)
    sigma = _ep_operands()["sigma"]
    s = _sgn(sgn, c.n, sigma)
    ref, A = dgrad64(c, ops.dy64, ops.w64) / s, dgrad64(c, ops.dy64.abs(), ops.w64.abs()) / s.abs()
    acc = acc_bound(A, k_len(c, True))

    def one(cfg):
        got = run_dgrad(lib, ops, sigma=sigma, sigma_group_n=sgn)
        _report(f"EP dgrad sigma/{sgn} {cfg}", check_bound(_nchw(got), ref, acc, f"dgrad sigma_group_n={sgn} {cfg}"))
    with_forms(c, True, one)


def _lrelu(t, slope):
    return torch.where(t > 0, t, t * slope)


def _bf16_range(t_lo, t_hi, residual, slope):
    """Bounds of bf16(lrelu(bf16(t) + residual)) in fp32 arithmetic (the header's order) over t in [t_lo, t_hi]: every
    step is monotone, so the kernel's result lies between the values at the two ends."""
    def at(t):
        f = t.float().to(torch.bfloat16).float() + residual.float()
        return _lrelu(f, torch.tensor(slope, dtype=torch.float32)).to(torch.bfloat16).double()
    return at(t_lo), at(t_hi)


INF_EP = ["act", "residual_act", "residual_y2", "y2"]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", INF_EP)
def test_inference_epilogue_every_form_vs_fp64(lib, variant):
    """The BatchNorm-folded sampling epilogue (VgConvEpilogue): t = conv / sigma + bias, [y = bf16(t) + residual],
    y = leaky_relu(., act_slope) stored as bf16, y2 = leaky_relu(post_scale y + post_shift, post_slope) from y as stored."""
    c = EP
    ops = Operands(c, seed=7)
    e = _ep_operands()
    g = torch.Generator(device=dev()).manual_seed(12)
    ho, wo = c.out_hw
    use_res = variant.startswith("residual")
    use_y2 = variant.endswith("y2")
    slope = 1.0 if variant == "y2" else 0.2
    residual = (2 * torch.randn(c.n, ho, wo, c.cout, generator=g, device=dev())).to(torch.bfloat16) if use_res else None
    post = (torch.rand(c.cout, generator=g, device=dev()) + 0.5, 0.3 * torch.randn(c.cout, generator=g, device=dev()), 0.1)
    bias, sigma = e["bias"], e["sigma"]
    s = _sgn(0, c.n, sigma)
    t = fwd64(c, ops.x64, ops.w64) / s + bias.double().view(1, -1, 1, 1)
    A = fwd64(c, ops.x64.abs(), ops.w64.abs()) / s.abs() + bias.double().abs().view(1, -1, 1, 1)
    acc = acc_bound(A, k_len(c, False))

    def one(cfg):
        out = run_forward(lib, ops, bias=bias, sigma=sigma, act_slope=slope, residual=residual, y2=use_y2,
                          post=post if use_y2 else None)
        y, y2 = out if use_y2 else (out, None)
        y = _nchw(y)
        tag = f"inference {variant} {cfg}"
        if use_res:
            lo, hi = _bf16_range(t - acc, t + acc, _nchw(residual), slope)
            yd = y.double()
            bad = (yd < lo) | (yd > hi)
            assert not bad.any(), f"{tag}: {int(bad.sum())} elements outside [lo, hi] at {_where(bad)}"
        else:
            _report(tag, check_bound(y, _lrelu(t, slope), acc * max(slope, 1.0), tag))
        if use_y2:
            ps, pt, pslope = post
            # the second output from y AS STORED: fp32 fma(post_scale, y, post_shift), leaky_relu, round
            a = (ps.double().view(1, -1, 1, 1) * y.double() + pt.double().view(1, -1, 1, 1)).float()
            ref2 = _lrelu(a, torch.tensor(pslope, dtype=torch.float32)).double()
            check_bound(_nchw(y2), ref2, torch.zeros_like(ref2), tag + " y2", half_ulp_frac=0.999)
    with_forms(c, False, one)


@pytest.mark.gpu
def test_fused_epilogue_rejects_unsupported_combinations(lib):
    """act_slope / residual / y2 need a bf16 output with c_out % 64 == 0 on the tensor-core path: VG_EUNSUPPORTED
    (never a silently different epilogue) for an fp32 output, a single output channel, and the CUDA-core path."""
    c = EP
    ops = Operands(c, seed=8)
    ho, wo = c.out_hw
    res = torch.zeros(c.n, ho, wo, c.cout, dtype=torch.bfloat16, device=dev())
    ps, pt = torch.ones(c.cout, device=dev()), torch.zeros(c.cout, device=dev())
    for kw in (dict(act_slope=0.2), dict(residual=res), dict(y2=True, post=(ps, pt, 1.0))):
        assert run_forward(lib, ops, torch.float32, raw=True, **kw) == VG_EUNSUPPORTED, kw
        prev = lib.load().vg_set_force_simt(1)
        try:
            assert run_forward(lib, ops, raw=True, **kw) == VG_EUNSUPPORTED, ("CUDA-core path", kw)
        finally:
            lib.load().vg_set_force_simt(prev)
    c1 = FORM_CASES["out1_20x12"]
    ops1 = Operands(c1, seed=9)
    assert run_forward(lib, ops1, raw=True, act_slope=0.2) == VG_EUNSUPPORTED
    torch.cuda.synchronize()


# ---- 4. weight gradient ------------------------------------------------------------------------------------------------
WGRAD_CASES = {
    # name: (case, workspace, accumulate into a non-zero dw, dbias)
    "nb1_3x3_cs64_nonsq": (Case(3, 64, 64, 20, 12, 3, 1, 1), True, False, True),       # c_u 64, 9 slabs (odd)
    "nb2_s2_nonsq": (Case(2, 128, 128, 24, 16, 3, 2, 1), True, True, False),           # c_u 128, stride-2 parity maps
    "nb4_256_1split": (Case(1, 64, 256, 8, 8, 3, 1, 1), True, False, False),           # c_u 256, one box: one split
    "nb4_512_many": (Case(8, 512, 512, 12, 10, 3, 1, 1), True, False, False),          # c_u 512, many splits
    "1x1_unpacked": (Case(4, 128, 256, 16, 24, 1, 1, 0), True, True, False),           # 1x1: torch layout, no unpack
    "1x1_s2": (Case(3, 256, 128, 16, 12, 1, 2, 0), True, False, False),
    "tr4x4": (Case(3, 256, 128, 12, 8, 4, 2, 1, 1), True, False, True),                # c_u = c_in (transposed)
    "3x3_no_ws": (Case(3, 64, 128, 20, 12, 3, 1, 1), False, True, False),              # k > 1, null workspace
    "tr4x4_no_ws": (Case(2, 128, 64, 8, 12, 4, 2, 1, 1), False, False, False),
    "big_batch": (Case(32, 64, 64, 48, 48, 3, 1, 1), True, True, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WGRAD_CASES))
def test_wgrad_vs_fp64(lib, name):
    c, use_ws, accumulate, use_db = WGRAD_CASES[name]
    ops = Operands(c, seed=_seed(name) + 17)
    g = torch.Generator(device=dev()).manual_seed(3)
    dw0 = torch.randn(c.wshape(), generator=g, device=dev()) * 0.01 if accumulate else torch.zeros(c.wshape(), device=dev())
    dw = dw0.clone()
    db = torch.zeros(c.cout, device=dev()) if use_db else None
    ws = torch.full((dw.numel(),), float("nan"), device=dev()) if use_ws else None
    d = _desc(c)
    lib.call("vg_conv_wgrad", C.byref(d), ops.x.data_ptr(), ops.dy.data_ptr(), dw.data_ptr(),
             None if db is None else db.data_ptr(), None if ws is None else ws.data_ptr(), lib.stream_ptr())
    ref = wgrad64(c, ops.x64, ops.dy64) + dw0.double()
    A = wgrad64(c, ops.x64.abs(), ops.dy64.abs()) + dw0.double().abs()
    ho, wo = c.out_hw
    K = c.n * (ho * wo if not c.tr else c.h * c.w)           # pixels of the side the reduction runs over
    _report(f"wgrad {name}", check_bound(dw, ref, acc_bound(A, K), f"wgrad {name}"))
    if db is not None:
        check_bound(db, ops.dy64.sum((0, 2, 3)), acc_bound(ops.dy64.abs().sum((0, 2, 3)), c.n * ho * wo), f"dbias {name}")


# ---- 5. CUDA-core kernels ----------------------------------------------------------------------------------------------
SIMT_CASES = {
    # name: (case, act dtype, sigma_group_n or None)  - forward, dgrad and wgrad through the CUDA-core kernels
    "direct_s1_10x6": (Case(3, 6, 10, 10, 6, 3, 1, 1), torch.bfloat16, 1),
    "direct_s2_12x8": (Case(3, 6, 10, 12, 8, 3, 2, 1), torch.float32, 2),
    "direct_tr_6x4": (Case(3, 6, 10, 6, 4, 4, 2, 1, 1), torch.bfloat16, None),
    "direct_v8_9x7": (Case(2, 16, 24, 9, 7, 3, 1, 1), torch.float32, 1),
    "tc_shape_forced": (Case(3, 64, 128, 20, 12, 3, 1, 1), torch.bfloat16, 2),
    "expand1_strip_10x16": (Case(3, 1, 64, 10, 16, 3, 1, 1), torch.bfloat16, None),     # width % 8 == 0: strip kernels
    "expand1_12x10": (Case(3, 1, 64, 12, 10, 3, 1, 1), torch.bfloat16, None),           # width % 8 != 0
    "expand1_strip_f32": (Case(2, 1, 16, 6, 24, 3, 1, 1), torch.float32, None),
    "reduce1_10x16": (Case(3, 64, 1, 10, 16, 3, 1, 1), torch.bfloat16, None),
    "reduce1_12x10_f32": (Case(2, 64, 1, 12, 10, 3, 1, 1), torch.float32, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SIMT_CASES))
def test_cuda_core_kernels_vs_fp64(lib, name):
    c, adt, sgn = SIMT_CASES[name]
    ops = Operands(c, seed=_seed(name) + 23, act_dtype=adt)
    sigma = torch.tensor([1.3, 0.7, 2.2], device=dev()) if sgn is not None else None
    s = _sgn(sgn or 0, c.n, sigma) if sigma is not None else 1.0
    sa = s.abs() if sigma is not None else 1.0
    prev = lib.load().vg_set_force_simt(1)
    try:
        y = run_forward(lib, ops, adt, sigma=sigma, sigma_group_n=sgn or 0)
        dx = run_dgrad(lib, ops, sigma=sigma, sigma_group_n=sgn or 0)
        dw = torch.zeros(c.wshape(), device=dev())
        lib.call("vg_conv_wgrad", C.byref(_desc(c, adt, adt)), ops.x.data_ptr(), ops.dy.data_ptr(), dw.data_ptr(), None, None,
                 lib.stream_ptr())
    finally:
        lib.load().vg_set_force_simt(prev)
    ho, wo = c.out_hw
    r = check_bound(_nchw(y), fwd64(c, ops.x64, ops.w64) / s, acc_bound(fwd64(c, ops.x64.abs(), ops.w64.abs()) / sa, k_len(c, False)),
                    f"{name} forward")
    _report(f"simt {name} fwd {adt}", r)
    r = check_bound(_nchw(dx), dgrad64(c, ops.dy64, ops.w64) / s,
                    acc_bound(dgrad64(c, ops.dy64.abs(), ops.w64.abs()) / sa, k_len(c, True)), f"{name} dgrad")
    _report(f"simt {name} dgrad {adt}", r)
    K = c.n * (ho * wo if not c.tr else c.h * c.w)
    r = check_bound(dw, wgrad64(c, ops.x64, ops.dy64), acc_bound(wgrad64(c, ops.x64.abs(), ops.dy64.abs()), K), f"{name} wgrad")
    _report(f"simt {name} wgrad {adt}", r)


# ---- 6. every kernel instance runs -------------------------------------------------------------------------------------
TC_INSTANCES = (
    [("tc_conv_kernel", (bn, st, inf)) for bn, st in ((64, 4), (128, 3), (256, 4)) for inf in (0, 1)]
    + [("tc_conv_persist_kernel", a + (inf,)) for a in ((64, 4, 3, 4), (128, 2, 4, 8), (256, 1, 4, 8)) for inf in (0, 1)]
    + [("tc_conv_pair_kernel", a + (inf,)) for a in ((64, 4, 3, 4), (128, 2, 4, 8), (256, 1, 6, 8)) for inf in (0, 1)]
    + [("tc_wgrad_kernel", a) for a in ((1, 6), (2, 5), (4, 4))]
)


def _instances(names):
    """{(kernel, template arguments)} from demangled kernel names; bools print as true/false or (bool)0/1."""
    out = set()
    for nm in names:
        m = re.search(r"(tc_conv_kernel|tc_conv_persist_kernel|tc_conv_pair_kernel|tc_wgrad_kernel)<([^>]*)>", nm)
        if m:
            args = tuple(int({"true": "1", "false": "0"}.get(a, a).replace("(bool)", "")) for a in
                         (s.strip() for s in m.group(2).split(",")))
            out.add((m.group(1), args))
        if "wgrad_unpack_kernel" in nm:
            out.add(("wgrad_unpack_kernel", ()))
    return out


def test_instance_name_parser():
    names = ["void vg::tc_conv_kernel<64, 4, false>(vg::TcConvParams)", "void vg::tc_conv_pair_kernel<256, 1, 6, 8, (bool)1>(x)",
             "vg::wgrad_unpack_kernel(const float*, int, int, int, float*)"]
    assert _instances(names) == {("tc_conv_kernel", (64, 4, 0)), ("tc_conv_pair_kernel", (256, 1, 6, 8, 1)),
                                 ("wgrad_unpack_kernel", ())}
    assert len(set(TC_INSTANCES)) == 21


@pytest.mark.gpu
def test_every_tensor_core_kernel_instance_runs(lib):
    """One representative launch per kernel instance under torch.profiler: all 18 tc_conv_* instances (3 forms x 3 N tiles
    x training / inference epilogue), the three tc_wgrad_kernel instances and wgrad_unpack_kernel appear."""
    from torch.profiler import ProfilerActivity, profile
    c = EP
    ops = Operands(c, seed=10)
    e = _ep_operands()
    ps, pt = torch.ones(c.cout, device=dev()), torch.zeros(c.cout, device=dev())
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for inf in (False, True):
            def one(cfg):
                if inf:
                    run_forward(lib, ops, bias=e["bias"], act_slope=0.2, y2=True, post=(ps, pt, 0.5))
                else:
                    run_forward(lib, ops, bias=e["bias"])
            with_forms(c, False, one)
        for wc in ("nb1_3x3_cs64_nonsq", "nb2_s2_nonsq", "nb4_256_1split"):
            cw = WGRAD_CASES[wc][0]
            o = Operands(cw, seed=1)
            dw = torch.zeros(cw.wshape(), device=dev())
            ws = torch.empty(dw.numel(), device=dev())
            lib.call("vg_conv_wgrad", C.byref(_desc(cw)), o.x.data_ptr(), o.dy.data_ptr(), dw.data_ptr(), None, ws.data_ptr(),
                     lib.stream_ptr())
        torch.cuda.synchronize()
    names = [evt.name for evt in prof.events() if evt.device_type == torch.autograd.DeviceType.CUDA]
    if not names:
        pytest.skip("the profiler returned no CUDA kernel events on this machine")
    seen = _instances(names)
    want = set(TC_INSTANCES) | {("wgrad_unpack_kernel", ())}
    print("launched kernel instances:")
    for kname, args in sorted(seen):
        print(f"  {kname}<{', '.join(map(str, args))}>")
    missing = want - seen
    assert not missing, f"{len(missing)} of {len(want)} kernel entries never launched: {sorted(missing)}"
