#!/usr/bin/env python
"""Benchmark of the VAE-GAN training iteration (BASELINE.json metric: train images/s at 96x96,
global batch 256, on 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--global-batch B] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one full training iteration (G fwd, D(real), D(fake), D bwd + Adam, D(fake) again,
G bwd + Adam) on one synthetic batch.  N > 1 is launched by torchrun (one rank per GPU, NCCL):
the global batch is split over the ranks (strong scaling), BatchNorm statistics and gradients are
all-reduced.  Prints ONE JSON line on rank 0.  Every timed loop runs exactly K steps.

`value`  : whole-job images/s with the batch already resident in HBM (CUDA-graph replay).
`e2e`    : same metric through the public API with HOST batches: pinned H2D copy of every batch and a
           D2H read of the step's losses inside the timed region.
`roofline`: the dominant kernel (tcgen05 implicit-GEMM conv) on the hottest layer shape, timed alone
           with CUDA events: algorithmic FLOPs / duration vs the measured bf16 peak.
`cpu_baseline`: the oracle (a port of the reference's PyTorch CPU path) on the host cores, bounded.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch

IMAGE = 96
FEATURE = 64
GFLOP_PER_IMG_STEP = 127.59        # 3*G + 8*D forward GFLOPs, SURVEY.md section 8d / BASELINE.md
# algorithmic bytes of the memory-bound family per image per step (BASELINE.md section 3: 10 B x E_G + 30 B x E_D)
# and of the fused optimizer per step (28 B/param)
MB_PER_IMG_STEP = 270.0
OPT_GB_PER_STEP = 0.80


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(bf16=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ----------------------------------------------------------------------------------------------
def cpu_baseline(budget_s: float = 20.0, batch: int = 4):
    """The reference's CPU path (oracle port: same modules, BCE + Adam step the GPU parity tests use)
    on the host cores, bounded to ~budget_s.  TEST/CHECKER code: reported, never shipped."""
    from oracle import vaegan_oracle as O
    spec_g = O.GeneratorSpec(depth=2, length=1, feature_size=FEATURE)
    spec_d = O.DiscriminatorSpec(input_size=IMAGE)
    Pg, Pd = O.make_generator_params(spec_g, 0), O.make_discriminator_params(spec_d, 1)
    og, od = O.OptState(), O.OptState()
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(batch, 1, IMAGE, IMAGE, generator=g)
    O.train_step(Pg, Pd, og, od, x, spec_g, spec_d)            # warm-up
    t0, n = time.time(), 0
    while True:
        O.train_step(Pg, Pd, og, od, x, spec_g, spec_d)
        n += 1
        if time.time() - t0 > budget_s or n >= 8:
            break
    dt = time.time() - t0
    return {"value": round(batch * n / dt, 4), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} iterations of oracle.train_step (BCE + Adam, dropout/noise from torch RNG) at batch {batch}, "
                      f"1x{IMAGE}x{IMAGE}, after 1 warm-up; {dt / n:.2f} s/iteration"}


def gpu_lib_baseline(dev, batches=(256, 64), steps: int = 6, warm: int = 3):
    """The bar SURVEY.md section 2.1 / BASELINE.md section 4 name ("GPU-lib"): the SAME modules in stock PyTorch
    eager on this B200 - cuDNN convolutions, cuBLAS Linear layers, ATen BatchNorm / optimizer maths - i.e. what the
    reference notebook itself runs when `device = cuda:0` (README.md:694, 910-911).  CHECKER code (the oracle port
    on CUDA tensors; never imported by the product).  Full BCE + Adam iteration per step, CUDA events.
    Variants: fp32 with TF32 off (the notebook's default numerics), fp32 with TF32 on, bf16 autocast + channels_last."""
    from oracle import vaegan_oracle as O
    spec_g = O.GeneratorSpec(depth=2, length=1, feature_size=FEATURE)
    spec_d = O.DiscriminatorSpec(1, FEATURE, (1, 1, 1), (1, 2, 2), (2 * FEATURE, 4 * FEATURE, 8 * FEATURE), input_size=IMAGE)
    out = {}
    old_tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True

    def run(variant, batch):
        cl = variant == "bf16_autocast_channels_last"
        tf32 = variant != "fp32"
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32
        Pg = {k: v.to(dev) for k, v in O.make_generator_params(spec_g, 0).items()}
        Pd = {k: v.to(dev) for k, v in O.make_discriminator_params(spec_d, 1).items()}
        if cl:
            for P in (Pg, Pd):
                for k, v in P.items():
                    if v.dim() == 4:
                        P[k] = v.contiguous(memory_format=torch.channels_last)
        og, od = O.OptState(), O.OptState()
        g = torch.Generator().manual_seed(1234)
        x = torch.rand(batch, 1, IMAGE, IMAGE, generator=g).to(dev)
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)

        def one():
            if cl:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    return O.train_step(Pg, Pd, og, od, x, spec_g, spec_d)
            return O.train_step(Pg, Pd, og, od, x, spec_g, spec_d)

        for _ in range(warm):
            one()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        return {"images_per_s": round(batch / ms * 1e3, 1), "ms_per_step": round(ms, 2)}

    try:
        for batch in batches:
            for variant in ("fp32", "fp32_tf32", "bf16_autocast_channels_last"):
                key = f"{variant}_b{batch}"
                try:
                    out[key] = run(variant, batch)
                except torch.cuda.OutOfMemoryError:
                    out[key] = {"error": "out of memory"}
                except Exception as e:      # pragma: no cover - report, never fail the bench line
                    out[key] = {"error": f"{type(e).__name__}: {str(e)[:120]}"}
                torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark = old_tf32
    # `value` = the fastest library variant at the bench's own batch (batches[0]); the other batch is reported beside it
    good = {k: v["images_per_s"] for k, v in out.items() if "images_per_s" in v and k.endswith(f"_b{batches[0]}")}
    best = max(good, key=good.get) if good else None
    return {"kind": "stock PyTorch eager on the same B200 (cuDNN/cuBLAS/ATen), oracle port on CUDA tensors, "
                    "full BCE + Adam iteration, CUDA events", "unit": "images/s", "steps": steps, "warmup": warm,
            "variants": out, "best": best, "value": good.get(best) if best else None,
            "torch": torch.__version__, "cudnn": torch.backends.cudnn.version()}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port; the
    notebook itself is not present on the GPU box), all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use the host's cores
    try:
        torch.set_num_threads(max(1, min(len(os.sched_getaffinity(0)), 64)))
    except Exception:
        pass
    from oracle import vaegan_oracle as O
    batch = 4
    spec_g = O.GeneratorSpec(depth=2, length=1, feature_size=FEATURE)
    spec_d = O.DiscriminatorSpec(input_size=IMAGE)
    Pg, Pd = O.make_generator_params(spec_g, 0), O.make_discriminator_params(spec_d, 1)
    og, od = O.OptState(), O.OptState()
    g = torch.Generator().manual_seed(1234)
    xs = [torch.rand(batch, 1, IMAGE, IMAGE, generator=g) for _ in range(2)]
    steps = args.steps
    warm = max(1, min(args.warmup, 1))
    for i in range(warm):
        O.train_step(Pg, Pd, og, od, xs[i % 2], spec_g, spec_d)
    t0 = time.time()
    for i in range(steps):
        O.train_step(Pg, Pd, og, od, xs[i % 2], spec_g, spec_d)
    dt = time.time() - t0
    val = batch * steps / dt
    sample = (f"each step = one oracle.train_step (BCE + Adam) on a bounded sample of {batch} images of the "
              f"global-batch-{args.global_batch} workload; {steps} steps after {warm} warm-up")
    print(json.dumps({
        "impl": "reference", "metric": "train_images_per_sec", "value": round(val, 4), "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": round(1000 * dt / steps, 2),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"VAE-GAN train step 1x{IMAGE}x{IMAGE}, depth 2 / length 1 / feature_size {FEATURE}, "
                               f"global batch {args.global_batch} (CPU arm: {batch}-image sample per step)",
                   "global_batch": args.global_batch, "parallelism": "cpu"},
        "cpu_baseline": {"value": round(val, 4), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(val, 4), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------
def roofline_probe(dev, batch: int, peaks):
    """Dominant kernel = tc_conv_kernel.  Hottest layer of the step: D res0.conv2, Conv2d 128->128
    3x3 s1 at 96x96 (2.718 GFLOP/img forward; SURVEY.md Appendix A).  Timed alone, CUDA events on the
    launching stream; the 128-channel activation is batch*96*96*128*2 B (>= 150 MB at batch 64) so
    every launch streams its input from HBM, not from the 126 MB L2."""
    import vae_gan_b200.functional as VF
    cin = cout = 128
    g = torch.Generator().manual_seed(0)
    nbuf = 3
    xs = [VF.as_act(torch.randn(batch, cin, IMAGE, IMAGE, generator=g).to(dev), torch.bfloat16) for _ in range(nbuf)]
    w = (torch.randn(cout, cin, 3, 3, generator=g) / 34.0).to(dev)
    geom = VF.ConvGeom(3, 1, 1, False)
    with torch.no_grad():
        for i in range(3):
            VF.conv(xs[i % nbuf], w, None, geom=geom)
        torch.cuda.synchronize(dev)
        # time ONLY the conv kernel: pack once, call the C ABI directly
        import ctypes as C
        from vae_gan_b200 import _lib
        d, ho, wo = VF._conv_desc(xs[0].shape, cout, geom, torch.bfloat16, torch.bfloat16)
        pk = torch.empty(w.numel(), dtype=torch.bfloat16, device=dev)
        pn = torch.empty(w.numel(), dtype=torch.bfloat16, device=dev)
        _lib.call("vg_conv_pack_weights", C.byref(d), w.data_ptr(), None, pk.data_ptr(), pn.data_ptr(), _lib.stream_ptr())
        y = VF.empty_act(batch, cout, ho, wo, torch.bfloat16, dev)
        iters = 12
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for i in range(iters):
            evs[i][0].record()
            _lib.call("vg_conv_forward", C.byref(d), xs[i % nbuf].data_ptr(), pk.data_ptr(), pn.data_ptr(), None, None,
                      y.data_ptr(), None, _lib.stream_ptr())
            evs[i][1].record()
        torch.cuda.synchronize(dev)
    ms = sorted(a.elapsed_time(b) for a, b in evs)
    avg = sum(ms[1:-1]) / (len(ms) - 2)
    flops = 2.0 * batch * IMAGE * IMAGE * cout * cin * 9
    achieved = flops / (avg * 1e-3) / 1e12
    traffic = ncu_traffic("conv_128x128_fwd", batch)       # measured by ncu this round, or None
    return {"bound": "tensor", "achieved": round(achieved, 1), "peak": peaks["bf16"], "unit": "TFLOP/s",
            "frac": round(achieved / peaks["bf16"], 4), "traffic": traffic,
            "kernel": "tc_conv_pair_kernel<128,2,4,8> (persistent cta_group::2 tcgen05 implicit GEMM), Conv2d 128->128 3x3 s1 @96x96",
            "batch": batch, "ms_per_launch": round(avg, 4), "flop_per_launch": flops,
            "peak_source": f"{peaks['source']} bf16 burst (kernel timed alone)"}


def roofline_hbm_probe(dev, batch: int, peaks):
    """Top memory-bound kernel of the step by time share: the BatchNorm(+LeakyReLU) backward APPLY
    (dx = gamma*rstd*(g - mean(g) - xhat*mean(g*xhat)), g = dy*lrelu'), on the 128-channel 96x96 tensor of D's first
    residual block.  Algorithmic bytes: read dy, read x, write dx at bf16 = 6 B/element (SURVEY.md section 8d).
    Timed alone with CUDA events; three rotating buffer sets (> 126 MB L2 each)."""
    import ctypes as C
    import vae_gan_b200.functional as VF
    from vae_gan_b200 import _lib
    c = 128
    g = torch.Generator().manual_seed(0)
    nbuf = 3
    xs = [VF.as_act(torch.randn(batch, c, IMAGE, IMAGE, generator=g).to(dev), torch.bfloat16) for _ in range(nbuf)]
    dys = [VF.as_act(torch.randn(batch, c, IMAGE, IMAGE, generator=g).to(dev), torch.bfloat16) for _ in range(nbuf)]
    dx = torch.empty_like(xs[0])
    gamma = torch.rand(c, device=dev) + 0.5
    beta = torch.randn(c, device=dev) * 0.1
    mr = torch.cat([torch.zeros(c, device=dev), torch.ones(c, device=dev)])
    sums = torch.zeros(2 * c, dtype=torch.float64, device=dev)
    d = VF._bn_desc(xs[0], 0.2, 0.0, 0, True)
    rows = batch * IMAGE * IMAGE
    iters = 12
    s = _lib.stream_ptr()
    for i in range(3):
        _lib.call("vg_bn_act_backward_apply", dys[i % nbuf].data_ptr(), xs[i % nbuf].data_ptr(), mr.data_ptr(), gamma.data_ptr(),
                  beta.data_ptr(), sums.data_ptr(), float(rows), C.byref(d), None, None, dx.data_ptr(), s)
    torch.cuda.synchronize(dev)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for i in range(iters):
        evs[i][0].record()
        _lib.call("vg_bn_act_backward_apply", dys[i % nbuf].data_ptr(), xs[i % nbuf].data_ptr(), mr.data_ptr(), gamma.data_ptr(),
                  beta.data_ptr(), sums.data_ptr(), float(rows), C.byref(d), None, None, dx.data_ptr(), s)
        evs[i][1].record()
    torch.cuda.synchronize(dev)
    ms = sorted(a.elapsed_time(b) for a, b in evs)
    avg = sum(ms[1:-1]) / (len(ms) - 2)
    nbytes = 3.0 * rows * c * 2
    achieved = nbytes / (avg * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm"], "unit": "GB/s",
            "frac": round(achieved / peaks["hbm"], 4), "traffic": ncu_traffic("bn_act_bwd_apply", batch),
            "kernel": "BatchNorm+LeakyReLU backward apply (vg_bn_act_backward_apply), 128 channels @96x96",
            "batch": batch, "ms_per_launch": round(avg, 4), "bytes_per_launch": nbytes,
            "peak_source": f"{peaks['source']} HBM copy bandwidth"}


def ncu_traffic(tag: str, batch: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture
    of this round (profiles/r2_ncu_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep); None when
    no capture of that kernel at that batch is committed."""
    f = ROOT / "profiles" / "r2_ncu_traffic.json"
    if not f.exists():
        return None
    try:
        d = json.loads(f.read_text())
        e = d.get(tag)
        if e and int(e.get("batch", -1)) == int(batch):
            return float(e["dram_bytes"])
    except Exception:
        pass
    return None


DUMP_MAX_ELEMS = 1 << 21        # 8 MB of float32 per array; the five large arrays stay well under 64 MB in all


def dump_outputs(out_dir, losses, tr, G, D):
    """--dump-outputs: what the last timed step handed its caller, one float32 DIR/<name>.npy per array - the step's
    losses as read_losses() returns them (summed over the ranks), its reconstruction `gen`, latent `mu` / `log_var` and
    discriminator logits `d_real` / `d_fake` / `d_gen` (NCHW order; with several GPUs these per-sample arrays are rank 0's
    shard of the batch), and the trained networks as `G_state` / `D_state` (every floating-point state-dict entry,
    flattened and concatenated in state-dict order).  An array of more than DUMP_MAX_ELEMS elements is stored as its
    values at a fixed sample of flat indices (numpy default_rng(0), sorted), so two runs with the same arguments can be
    compared element for element."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {k: torch.tensor(v, dtype=torch.float32) for k, v in losses.items()}
    arrays.update(tr.last)
    for tag, net in (("G", G), ("D", D)):
        arrays[f"{tag}_state"] = torch.cat([v.detach().float().flatten() for v in net.state_dict().values()
                                            if v.is_floating_point()])
    total = 0
    for name, t in arrays.items():
        a = t.detach().float().contiguous().cpu().numpy()
        if a.size > DUMP_MAX_ELEMS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(out_dir / f"{name}.npy", a)
        total += a.nbytes
    assert total <= 64 << 20, f"--dump-outputs wrote {total} bytes"


def run_decode_sweep(args):
    """BASELINE.json config 5: decoder-only sampling, z ~ N(0, I) of shape (B, 256, 24, 24) -> 96x96 image,
    eval mode (BatchNorm running statistics, no dropout), batch 1..4096 on one GPU, CUDA-graph replay.
    `folded`: vae_gan_b200.sampling.FoldedGenerator (BatchNorms folded into the convolutions, activation / residual /
    next pre-activation in the tensor-core epilogue); `module`: the nn.Module's own eval-mode forward (un-folded).
    Also one encode() and one eval reconstruction point at batch 256 (README.md:655-659, 1223-1226)."""
    import vae_gan_b200 as V
    from vae_gan_b200.sampling import FoldedGenerator
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    rows = []

    def time_graph(fn, inp, iters):
        for _ in range(3):
            fn(inp)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            fn(inp)
        for _ in range(3):
            graph.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
        del graph
        return e0.elapsed_time(e1) / iters

    with V.compute_dtype(torch.bfloat16), torch.no_grad():
        G, _ = V.build_vae_gan(feature_size=FEATURE, image_size=IMAGE)
        G = G.to(dev).eval()
        G.set_is_training(False)
        fg = FoldedGenerator(G)
        for B in (1, 4, 16, 64, 256, 1024, 4096):
            z = torch.randn(B, 256, IMAGE // 4, IMAGE // 4, device=dev)
            iters = 20 if B <= 1024 else 8
            ms_f = time_graph(fg.decode, z, iters)
            ms_m = time_graph(G.decode, z, iters)
            rows.append({"batch": B, "ms": round(ms_f, 4), "images_per_s": round(B / ms_f * 1e3, 1),
                         "tflops": round(3.796e9 * B / (ms_f * 1e-3) / 1e12, 1),
                         "module_ms": round(ms_m, 4), "module_images_per_s": round(B / ms_m * 1e3, 1)})
        x = torch.rand(256, 1, IMAGE, IMAGE, device=dev)
        ms_enc = time_graph(fg.encode, x, 20)
        ms_rec = time_graph(fg.reconstruct, x, 20)
        ms_enc_m = time_graph(G.encode, x, 20)
    peaks = measured_peaks()
    best = max(rows, key=lambda r: r["images_per_s"])
    print(json.dumps({"metric": "decode_images_per_sec", "unit": "images/s", "n_gpus": 1, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": "decoder-only sampling sweep, latent (B,256,24,24) -> 1x96x96, eval mode, BatchNorm-folded "
                                             "FoldedGenerator (module = un-folded nn.Module eval forward), CUDA-graph replay"},
                      "sweep": rows, "value": best["images_per_s"], "higher_is_better": True,
                      "frac_of_tensor_peak": round(best["tflops"] / peaks["bf16"], 4),
                      "encode_b256": {"ms": round(ms_enc, 4), "images_per_s": round(256 / ms_enc * 1e3, 1), "module_ms": round(ms_enc_m, 4),
                                      "tflops": round((3.4186e9 + 0.6795e9) * 256 / (ms_enc * 1e-3) / 1e12, 1)},
                      "reconstruct_b256": {"ms": round(ms_rec, 4), "images_per_s": round(256 / ms_rec * 1e3, 1)}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--global-batch", type=int, default=256)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-lib-baseline", action="store_true", help="skip the stock-PyTorch-on-this-GPU leg (gpu_lib_baseline)")
    ap.add_argument("--fp32", action="store_true", help="run the fp32 parity path instead of bf16")
    ap.add_argument("--loss-mode", default="bce", choices=["bce", "wgan", "wgan_gp"],
                    help="bce + adam = BASELINE north_star (default); wgan_gp + --optimizer rmsprop = the notebook as written")
    ap.add_argument("--optimizer", default="adam", choices=["adam", "rmsprop"])
    ap.add_argument("--workload", default="train", choices=["train", "cfg4", "decode"],
                    help="train: BASELINE metric (96x96, fs 64); cfg4: 256x256, widths x2; decode: config-5 sampling sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs); "
                         "runs with deterministic (ordered) reductions so that runs with the same arguments match")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "decode"):
        ap.error("--dump-outputs applies to the training step of --impl ours (--workload train or cfg4)")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "decode":
        run_decode_sweep(args)
        return
    global IMAGE, FEATURE, GFLOP_PER_IMG_STEP, MB_PER_IMG_STEP, OPT_GB_PER_STEP
    if args.workload == "cfg4":
        IMAGE, FEATURE, GFLOP_PER_IMG_STEP = 256, 128, 3621.5
        MB_PER_IMG_STEP, OPT_GB_PER_STEP = 10 * 81.99 + 30 * 100.66, 28 * 305.13e6 / 1e9
        if args.global_batch == 256:
            args.global_batch = 16 * max(1, int(os.environ.get("WORLD_SIZE", "1")))

    import torch.distributed as dist
    import vae_gan_b200 as V

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    assert args.global_batch % world == 0
    local_b = args.global_batch // world
    W = max(args.warmup, 3)
    K = args.steps
    peaks = measured_peaks()
    cdt = torch.float32 if args.fp32 else torch.bfloat16
    if args.dump_outputs:
        # outputs meant for comparison need ordered cross-block sums: with the default atomics the last bits of a step vary
        # from run to run, and Adam's lr*sign(g) steps on near-zero gradients grow them into weights that differ by
        # percents within a few dozen steps.  Without --dump-outputs the default (atomic) path is timed.
        V.set_deterministic(True, dev)

    torch.manual_seed(0)
    with V.compute_dtype(cdt):
        G, D = V.build_vae_gan(feature_size=FEATURE, image_size=IMAGE)
        G, D = G.to(dev).train(), D.to(dev).train()
        tr = V.VaeGanTrainer(G, D, loss_mode=args.loss_mode, optimizer=args.optimizer, lr=3e-4, process_group=pg)
        V.config.sample_offset = rank * local_b
        g = torch.Generator().manual_seed(1234 + rank)
        n_host = 4
        host = [torch.rand(local_b, 1, IMAGE, IMAGE, generator=g).pin_memory() for _ in range(n_host)]
        x_dev = host[0].to(dev)
        if world > 1:
            t = torch.ones(1, device=dev)
            dist.all_reduce(t)          # initialise the NCCL communicator before any capture
        torch.cuda.synchronize(dev)

        mode = "eager"
        launches_per_step = None
        if not args.no_graph:
            try:
                for _ in range(2):
                    tr._step_impl(x_dev)
                torch.cuda.synchronize(dev)
                l0 = V._lib.launch_count()
                tr.capture(x_dev, warmup=1)
                mode = "cuda_graph"
                # capture() ran 1 eager step + 1 captured step
                launches_per_step = (V._lib.launch_count() - l0) // 2
            except Exception as e:      # pragma: no cover
                if rank == 0:
                    print(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); running eagerly", file=sys.stderr)
                tr.graph = None
                torch.cuda.synchronize(dev)
        if launches_per_step is None:
            l0 = V._lib.launch_count()
            tr._step_impl(x_dev)
            launches_per_step = V._lib.launch_count() - l0

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)

        # ---------------- device-resident throughput ----------------
        for _ in range(W):
            tr.step(x_dev if tr.graph is None else tr.static_real)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            tr.step(x_dev if tr.graph is None else tr.static_real)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop()
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        ms_per_step = ms / K
        value = args.global_batch * K / (ms * 1e-3)
        losses = tr.read_losses()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, losses, tr, G, D)

        # ---------------- end to end: host batches in, losses out, every step ----------------
        # Public API: InputPipeline (pinned staging + copy stream, double buffered: the H2D copy of batch k+1 runs under
        # step k) -> VaeGanTrainer.step -> read_losses (one D2H read of the step's scalars).
        def e2e_run(pipe, batches, n_steps):
            pipe.submit(batches[0])
            for i in range(2):
                xb = pipe.get()
                pipe.submit(batches[(i + 1) % len(batches)])
                tr.step(xb)
                pipe.release()
                tr.read_losses()
            barrier()
            e0.record()
            for i in range(n_steps):
                xb = pipe.get()                                       # this step's batch (copied while the previous step ran)
                pipe.submit(batches[(i + 3) % len(batches)])          # pinned H2D copy of the next step's batch
                tr.step(xb)
                pipe.release()
                tr.read_losses()                                      # D2H read of this step's scalars
            e1.record()
            barrier()
            t = e0.elapsed_time(e1)
            if world > 1:
                tt = torch.tensor([t], device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = float(tt)
            pipe.get()                                                # drain the last prefetch
            return t

        pipe = V.InputPipeline(dev, (local_b, 1, IMAGE, IMAGE), torch.float32, normalize=False)
        ms_e = e2e_run(pipe, host, K)
        e2e_value = args.global_batch * K / (ms_e * 1e-3)
        # the same with RAW 8-bit pixels: 1 B/pixel over PCIe, per-image min-max normalisation on the device (SURVEY N3)
        host_u8 = [(h * 255.0).round().to(torch.uint8).pin_memory() for h in host]
        pipe8 = V.InputPipeline(dev, (local_b, 1, IMAGE, IMAGE), torch.uint8, normalize=True)
        ms_e8 = e2e_run(pipe8, host_u8, K)
        e2e_u8 = args.global_batch * K / (ms_e8 * 1e-3)

        roof = roof_hbm = cpu = lib = None
        # drop the captured graph (it holds NCCL work) on EVERY rank before any teardown
        tr.graph = None
        torch.cuda.synchronize(dev)
        barrier()
        if rank == 0:
            torch.cuda.empty_cache()
            roof = roofline_probe(dev, min(local_b, 64), peaks)
            roof_hbm = roofline_hbm_probe(dev, min(local_b, 64), peaks)
            if world == 1 and not args.skip_lib_baseline and args.workload == "train":
                del tr, G, D
                torch.cuda.empty_cache()
                lib = gpu_lib_baseline(dev, batches=tuple(dict.fromkeys((args.global_batch, 64))))
            if world == 1 and not args.skip_cpu_baseline:
                cpu = cpu_baseline()

    if rank == 0:
        step_tflops = GFLOP_PER_IMG_STEP * 1e9 * args.global_batch / (ms_per_step * 1e-3) / 1e12 / world
        # step-level roofline (SURVEY.md section 8d): t_ideal = F_step / tensor peak + Bytes_step / HBM peak, per GPU
        t_tensor = GFLOP_PER_IMG_STEP * 1e9 * local_b / (peaks["bf16"] * 1e12) * 1e3
        t_hbm = (MB_PER_IMG_STEP * 1e6 * local_b + OPT_GB_PER_STEP * 1e9) / (peaks["hbm"] * 1e9) * 1e3
        out = {
            "metric": "train_images_per_sec", "value": round(value, 2), "unit": "images/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32" if args.fp32 else "bf16", "data": "synthetic",
            "config": {
                "workload": "full VAE-GAN train step (encoder+decoder+discriminator, KL + L1/MSE + " +
                            {"bce": "adversarial BCE", "wgan": "critic loss + clamp", "wgan_gp": "critic loss + 10 x gradient penalty "
                             "(double backward) + clamp"}[args.loss_mode] + f", {args.optimizer}), "
                            f"1x{IMAGE}x{IMAGE} images, depth 2 / length 1 / feature_size {FEATURE}, global batch "
                            f"{args.global_batch} ({local_b}/GPU), SyncBN + gradient all-reduce" + ("" if world > 1 else " (1 GPU: no collectives)"),
                "global_batch": args.global_batch, "per_gpu_batch": local_b, "parallelism": f"dp{world}", "mode": mode,
                "loss_mode": args.loss_mode, "optimizer": args.optimizer,
                "l2_note": "activations of one step (several GB) far exceed the 126 MB L2; no flush needed",
            },
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 2), "unit": "images/s", "h2d_bytes_per_step": local_b * IMAGE * IMAGE * 4 * world,
                    "d2h_bytes_per_step": 7 * 4 * world, "steps": K, "ms_per_step": round(ms_e / K, 3),
                    "api": "InputPipeline (pinned, copy stream, double buffered) -> VaeGanTrainer.step -> read_losses"},
            "e2e_u8_pipeline": {"value": round(e2e_u8, 2), "unit": "images/s", "h2d_bytes_per_step": local_b * IMAGE * IMAGE * world,
                                "d2h_bytes_per_step": 7 * 4 * world, "steps": K, "ms_per_step": round(ms_e8 / K, 3),
                                "note": "raw uint8 pixels over PCIe, vg_normalize_images (per-image min-max, float64 math) on the copy stream"},
            "gpu_launches": int(launches_per_step * K),
            "launches_per_step": int(launches_per_step),
            "step_model_tflops_per_gpu": round(step_tflops, 1),
            "step_frac_of_tensor_peak": round(step_tflops / peaks["bf16_sustained"], 4),
            "t_ideal_ms": round(t_tensor + t_hbm, 3), "t_ideal_tensor_ms": round(t_tensor, 3), "t_ideal_hbm_ms": round(t_hbm, 3),
            "t_measured_ms": round(ms_per_step, 3), "step_frac_of_ideal": round((t_tensor + t_hbm) / ms_per_step, 4),
            "roofline": roof,
            "roofline_hbm": roof_hbm,
            "gpu_lib_baseline": lib,
            "vs_gpu_lib": (round(value / lib["value"], 3) if lib and lib.get("value") else None),
            "cpu_baseline": cpu,
            "losses_last_step": {k: round(v, 4) for k, v in losses.items()},
        }
        if V.is_deterministic():
            out["config"]["reductions"] = "deterministic (ordered cross-block sums)"
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)       # skip NCCL/graph teardown ordering issues at interpreter exit


if __name__ == "__main__":
    main()
