#!/usr/bin/env python
"""Benchmark of the diffusion-sampling hot path (BASELINE.json metric: DDIM-50 voxels/s on the 3-D 160x224x160 UNet).

    python bench.py --gpus N --steps K --warmup W            # this repo's arm (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs, DIR/<name>.npy

Definitions (DESIGN.md section 4):
  * workload  = config C3 of BASELINE.json: DiffusionModelUNet 3-D (256, 256, 512), attention (F, F, T), heads
                (0, 0, 512), 2 res blocks, x = 1 x 1 x 160 x 224 x 160 per GPU, DDIMScheduler(1000,
                "scaled_linear_beta", 0.0005, 0.0195, clip_sample=False), random-init weights (zero-init convs
                redrawn N(0, 0.02^2)), synthetic noise — SURVEY.md section 8(d).
  * one STEP  = one DDIM iteration = UNet forward + scheduler.step on the per-GPU batch; all 50 iterations of a
                sample are identical work, so  value = n_gpus * voxels / (50 * seconds_per_step)  [voxels/s].
  * value     = inputs resident in HBM; e2e = the same metric through DiffusionInferer.sample() starting from pinned
                HOST noise (H2D), the per-step timestep H2D the reference API does, the final D2H of the sample and —
                at N > 1 — the all_gather of the finished samples.
  * roofline  = tensor-pipe: algorithmic FLOPs of the 3x3x3-conv launches of igemm_tc_kernel<256,6,pair> in the timed
                region / their CUDA-event time, against MEASURED_PEAKS.json's sustained bf16/fp16 GEMM throughput;
                roofline.secondary[] = the attention kernel (tensor) and the HBM-bound kernels (GroupNorm apply,
                DDIM step) timed the same way against the measured copy bandwidth.
  * other_configs = the other targets BASELINE.json names (C2 latent diffusion at batch 1 and 32, C4 VQVAE, C5
                ControlNet + classifier-free guidance), each with its wall clock through the public API, algorithmic
                TFLOP/s and (N = 1) the reference's CPU leg.
  * weak scaling: every GPU samples its own volume; the only collective is one all_gather of the finished samples.
  * reference arm / cpu_baseline: the unmodified reference installed under oracle/_ref (oracle/make_ref.sh; MONAI's
                layer wrappers come from oracle/monai_shim because MONAI is not installable offline), run through its
                own DiffusionInferer.sample on the host cores; the oracle port only if oracle/_ref is absent.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

C3 = dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(256, 256, 512),
          attention_levels=(False, False, True), num_head_channels=(0, 0, 512), num_res_blocks=2)
C3_SCHED = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0005, beta_end=0.0195,
                clip_sample=False)
C3_VOLUME = (160, 224, 160)
CPU_VOLUME = (32, 40, 32)       # the reference tutorial's volume: the full one cannot run on CPU (SURVEY.md section 8d)
DDIM_STEPS = 50
METRIC = "ddim50_voxels_per_s"

# the other BASELINE.json configurations (SURVEY.md section 8, "Benchmark model definitions")
C2_AEKL = dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(128, 128, 256), latent_channels=3,
               num_res_blocks=2, attention_levels=(False, False, False), with_encoder_nonlocal_attn=False,
               with_decoder_nonlocal_attn=False)
C2_UNET = dict(spatial_dims=2, in_channels=3, out_channels=3, num_res_blocks=2, num_channels=(128, 256, 512),
               attention_levels=(False, True, True), num_head_channels=(0, 256, 512))
C2_SCHED = dict(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0015, beta_end=0.0195)
C4_VQVAE = dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(256, 256), num_res_channels=256,
                num_res_layers=2, downsample_parameters=((2, 4, 1, 1),) * 2, upsample_parameters=((2, 4, 1, 1, 0),) * 2,
                num_embeddings=256, embedding_dim=32)
C5_COMMON = dict(spatial_dims=2, in_channels=3, num_res_blocks=1, num_channels=(128, 256, 256),
                 attention_levels=(False, True, True), num_head_channels=256, with_conditioning=True,
                 cross_attention_dim=1)
# algorithmic TFLOP (SURVEY.md section 8, table "Algorithmic work per UNet/AE forward": conv 2*N*V_out*Cin*Cout*k^d,
# attention 4*N*H*T*S*d, GEMM 2*M*N*K; no recomputation / padding / layout work)
TF_C3_FORWARD = 458.3
TF_C2_SAMPLE = 3.96          # 50 x 0.076 + decode 0.161, per sample
TF_C4_VOLUME = 8.95          # encode -> VQ -> decode of one 128^3 volume
TF_C5_STEP = 4.11            # ControlNet + UNet on the doubled batch, per guided sample and step


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        p = json.loads(f.read_text())
        return p.get("bf16_tflops_sustained", 1449.3), p.get("hbm_gbs", 6582.5), "measured"
    return 1400.0, 6650.0, "fallback"


def redraw_zero_params(m, seed=1):
    """Zero-init convolutions redrawn N(0, 0.02^2) so activations are non-degenerate (SURVEY.md section 8d)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in m.parameters():
            if p.numel() and float(p.abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    return m


def build_model_state(seed=0):
    """C3 UNet with the reference's parameter tree (constructed by this package: same keys and shapes)."""
    import torch
    from generativemodels_b200.networks.nets import DiffusionModelUNet
    torch.manual_seed(seed)
    return redraw_zero_params(DiffusionModelUNet(**C3).eval(), seed + 1)


# ---------------------------------------------------------------------------------------------------------------
# reference / CPU arm
# ---------------------------------------------------------------------------------------------------------------
REF_DIR = ROOT / "oracle" / "_ref"


def import_reference():
    """The unmodified reference from oracle/_ref (pip-installed by oracle/make_ref.sh) on top of the MONAI shim.
    Returns the `generative` package or None when it is not installed."""
    if not (REF_DIR / "generative" / "__init__.py").exists():
        return None
    mine = sys.modules.get("generative")
    if mine is not None and str(REF_DIR) not in str(getattr(mine, "__file__", "")):
        raise RuntimeError("this repository's `generative` alias is already imported in this process")
    try:
        import monai  # noqa: F401
    except Exception:
        sys.path.insert(0, str(ROOT / "oracle" / "monai_shim"))
    # ahead of the repository root, which carries this repo's own `generative` alias package
    sys.path.insert(0, str(REF_DIR))
    import generative  # noqa: F401
    import generative.inferers  # noqa: F401
    import generative.networks.nets  # noqa: F401
    import generative.networks.schedulers  # noqa: F401
    assert str(REF_DIR) in generative.__file__
    return generative


CPU_THREAD_CAP = 32


def cpu_threads():
    """One fixed policy for every CPU leg of every arm: min(host cores, 32) intra-op threads.  oneDNN's direct
    convolutions of these shapes run SLOWER on 64 threads across sockets than on 32 (round 1 measured 247 vs 411-460
    voxel/s on the same box when one leg auto-picked and the other took the default; round 2's default-64 run gave
    225) — a fixed cap keeps the legs comparable and the baseline at its better operating point."""
    import torch
    n = max(1, min(os.cpu_count() or 1, CPU_THREAD_CAP))
    if torch.get_num_threads() != n:
        torch.set_num_threads(n)
    return n


def cpu_c3_steps(state_dict, steps: int, warmup: int):
    """`steps` DDIM iterations of the C3 model at the tutorial volume on the host cores -> (voxels/s for DDIM-50,
    seconds per step, threads, kind)."""
    import torch
    ref = import_reference()
    cpu_threads()
    torch.manual_seed(1234)
    x = torch.randn(1, 1, *CPU_VOLUME)
    sd = {k: v.detach().cpu() for k, v in state_dict.items()}
    n = warmup + steps
    if ref is not None:
        from generative.inferers import DiffusionInferer
        from generative.networks.nets import DiffusionModelUNet
        from generative.networks.schedulers import DDIMScheduler
        m = DiffusionModelUNet(**C3).eval()
        m.load_state_dict(sd)
        sched = DDIMScheduler(**C3_SCHED)
        sched.set_timesteps(DDIM_STEPS)
        inferer = DiffusionInferer(sched)
        times = []
        orig_step = sched.step

        def timed_step(*a, **k):          # one timestamp per iteration of the reference's own sampling loop
            out = orig_step(*a, **k)
            times.append(time.perf_counter())
            return out
        sched.step = timed_step
        sched.timesteps = sched.timesteps[:n]
        t0 = time.perf_counter()
        with torch.no_grad():
            inferer.sample(input_noise=x, diffusion_model=m, scheduler=sched, verbose=False)
        stamps = [t0] + times
        per = [b - a for a, b in zip(stamps[:-1], stamps[1:])][warmup:]
        kind = "reference"
    else:
        from oracle import torch_oracle as O
        cfg = dict(num_head_channels=C3["num_head_channels"], norm_num_groups=32, norm_eps=1e-6, with_conditioning=False)
        sched = O.DDIMOracle(**C3_SCHED)
        sched.set_timesteps(DDIM_STEPS)
        per = []
        with torch.no_grad():
            for i, t in enumerate(sched.timesteps[:n]):
                t0 = time.perf_counter()
                eps = O.unet_forward(sd, cfg, x, torch.Tensor((t,)))
                x, _ = sched.step(eps, int(t), x)
                if i >= warmup:
                    per.append(time.perf_counter() - t0)
        kind = "port"
    sec = sum(per) / len(per)
    vox = CPU_VOLUME[0] * CPU_VOLUME[1] * CPU_VOLUME[2]
    return vox / (DDIM_STEPS * sec), sec, cpu_threads(), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model = build_model_state()
    value, sec, cores, kind = cpu_c3_steps(model.state_dict(), args.steps, args.warmup)
    what = ("the unmodified reference (oracle/_ref) through its DiffusionInferer.sample" if kind == "reference"
            else "oracle port of the reference CPU path (oracle/_ref absent)")
    sample = (f"{what}: UNet forward + DDIM step on 1x1x{'x'.join(map(str, CPU_VOLUME))} "
              f"(the full 160x224x160 volume needs ~60 GB of fp32 activations and 2x29.9 GiB attention scores on CPU), "
              f"{args.steps} steps after {args.warmup} warm-up, {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C3: 3D DiffusionModelUNet (256,256,512) DDIM-50", "volume": list(CPU_VOLUME),
                   "per_gpu_batch": 1},
        "cpu_baseline": {"value": value, "unit": "voxels/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def cpu_other_configs(states):
    """Bounded CPU legs of C2 / C4 / C5 through the reference (oracle/_ref), a few seconds each; None without it."""
    import torch
    if import_reference() is None:
        return {}
    cpu_threads()
    from generative.networks.nets import VQVAE, AutoencoderKL, ControlNet, DiffusionModelUNet
    from generative.networks.schedulers import DDIMScheduler
    out = {}
    with torch.no_grad():
        un = DiffusionModelUNet(**C2_UNET).eval(); un.load_state_dict(states["c2_unet"])
        ae = AutoencoderKL(**C2_AEKL).eval(); ae.load_state_dict(states["c2_ae"])
        s = DDIMScheduler(**C2_SCHED); s.set_timesteps(DDIM_STEPS)
        torch.manual_seed(1234)
        x = torch.randn(1, 3, 64, 64)
        ts = list(s.timesteps[:4])
        t0 = None
        for i, t in enumerate(ts):
            if i == 1:
                t0 = time.perf_counter()
            x, _ = s.step(un(x, timesteps=torch.Tensor((t,))), t, x)
        per_step = (time.perf_counter() - t0) / (len(ts) - 1)
        t0 = time.perf_counter()
        ae.decode_stage_2_outputs(x)
        dec = time.perf_counter() - t0
        sec = DDIM_STEPS * per_step + dec
        out["C2_ldm_n1"] = {"value": 1.0 / sec, "unit": "samples/s", "cores": cpu_threads(), "kind": "reference",
                            "sample": f"3 UNet+DDIM steps ({per_step:.2f} s each) x 50 + 1 decode ({dec:.2f} s)"}
        vq = VQVAE(**C4_VQVAE).eval(); vq.load_state_dict(states["c4"])
        xv = torch.rand(1, 1, 64, 64, 64)
        t0 = time.perf_counter()
        vq(xv)
        sec = time.perf_counter() - t0
        out["C4_vqvae"] = {"value": 64 ** 3 / sec, "unit": "voxels/s", "cores": cpu_threads(), "kind": "reference",
                           "sample": f"one encode->VQ->decode of 1x64^3 ({sec:.2f} s; the GPU leg runs 1x128^3)"}
        u5 = DiffusionModelUNet(out_channels=3, **C5_COMMON).eval(); u5.load_state_dict(states["c5_unet"])
        c5 = ControlNet(conditioning_embedding_in_channels=1, conditioning_embedding_num_channels=(16,),
                        **C5_COMMON).eval(); c5.load_state_dict(states["c5_cn"])
        x2 = torch.randn(2, 3, 256, 256)
        ctx = torch.cat([-torch.ones(1, 1, 1), torch.ones(1, 1, 1)])
        t0 = time.perf_counter()
        down, mid = c5(x=x2, timesteps=torch.Tensor((500,)), controlnet_cond=c5_mask().expand(2, -1, -1, -1), context=ctx)
        u5(x2, timesteps=torch.Tensor((500,)), context=ctx, down_block_additional_residuals=down,
           mid_block_additional_residual=mid)
        sec = time.perf_counter() - t0
        out["C5_controlnet_cfg"] = {"value": 1.0 / (DDIM_STEPS * sec), "unit": "guided samples/s", "cores": cpu_threads(),
                                    "kind": "reference", "sample": f"1 of 50 guided steps ({sec:.1f} s), scaled"}
    return out


def c5_mask():
    import torch
    yy, xx = torch.meshgrid(torch.arange(256), torch.arange(256), indexing="ij")
    return (((xx - 128) ** 2 + (yy - 128) ** 2) < 100 ** 2).float()[None, None]


# ---------------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower() == "active" for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


KERNELS_PER_CALL = {"b200_groupnorm_stats": 2}
NOT_KERNELS = ("b200_last_error_string", "b200_version", "b200_act_dtype", "b200_device_check", "b200_sm_count",
               "b200_abi_sizeof", "b200_groupnorm_workspace_bytes", "b200_attention_flash_workspace_bytes",
               "b200_igemm_split_workspace_bytes")


class Instrument:
    """Launch counter over every C-ABI entry point + CUDA events (on the launching stream = torch's current stream)
    around the kernels that carry a roofline entry.  Active only between start() and stop()."""

    def __init__(self, lib, ops, _lib):
        import ctypes as C
        import torch
        self.torch, self.ops, self.on, self.n = torch, ops, False, 0
        self.ev = {k: [] for k in ("conv", "attn", "gn_apply", "ddim")}
        self.work = {k: 0.0 for k in self.ev}           # FLOPs (conv, attn) or bytes (gn_apply, ddim)
        for name in _lib.SIGNATURES:
            if name in NOT_KERNELS:
                continue
            fn = getattr(lib, name)
            setattr(lib, name, self._wrap(name, fn, KERNELS_PER_CALL.get(name, 1), C))
        self.raw_igemm = ops.igemm_raw
        ops.igemm_raw = self._igemm

    def _timed(self, key, work, call):
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record()
        r = call()
        e1.record()
        self.ev[key].append((e0, e1))
        self.work[key] += work
        return r

    def _wrap(self, name, fn, k, C):
        def counted(*a):
            if not self.on:
                return fn(*a)
            self.n += k
            if name == "b200_attention_flash":
                p = a[0]._obj
                return self._timed("attn", 4.0 * p.B * p.heads * p.T * p.S * p.dh, lambda: fn(*a))
            if name == "b200_groupnorm_apply":
                p = a[0]._obj
                ch = p.x_C[0] + (p.x_C[1] if p.x_ptr[1] else 0)
                return self._timed("gn_apply", 2.0 * 2 * p.N * p.spatial * ch, lambda: fn(*a))     # 1 read + 1 write, 2 B
            if name == "b200_ddim_step":
                return self._timed("ddim", 16.0 * a[6], lambda: fn(*a))       # eps + x read, x_prev + x0 written, fp32
            return fn(*a)
        return counted

    def _igemm(self, p):
        dominant = self.on and p.n_seg >= 27 and p.out_cols > 128              # 3x3x3 convs -> igemm_tc_kernel<256,4>
        if not dominant:
            return self.raw_igemm(p)
        rows = p.out_N * p.out_D * p.out_H * p.out_W
        kval = sum(min(p.a_C[p.seg[i].src] - p.seg[i].c0 * 64, p.seg[i].nchunks * 64) for i in range(p.n_seg))
        return self._timed("conv", 2.0 * rows * p.cout * kval, lambda: self.raw_igemm(p))

    def start(self):
        self.on, self.n = True, 0
        for k in self.ev:
            self.ev[k], self.work[k] = [], 0.0

    def stop(self):
        self.on = False

    def ms(self, key):
        return sum(a.elapsed_time(b) for a, b in self.ev[key])


DUMP_BYTES = 60 << 20          # of array data: with the .npy headers, under 64 MB (10^6 bytes) in all


def dump_outputs(outdir, arrays):
    """Write each tensor as <outdir>/<name>.npy in float32.  Past DUMP_BYTES in all, each one is cut to a fixed, seeded
    sample of its flattened elements (the same positions on every run), an equal share of DUMP_BYTES each."""
    import numpy as np
    import torch
    os.makedirs(outdir, exist_ok=True)
    total = sum(a.numel() * 4 for a in arrays.values())
    share = DUMP_BYTES // (4 * len(arrays))
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        if total > DUMP_BYTES and a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(outdir, f"{name}.npy"), a.numpy())


def time_calls(fn, n, sync):
    fn()
    sync()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    sync()
    return (time.perf_counter() - t0) / n


def other_configs_gpu(world, rank, peak_tf, states_out):
    """C2 (batch 1 and 32 per GPU), C4, C5 through the public API on this rank's GPU; per-GPU batches are fixed as N
    grows (weak scaling), times are the max over ranks."""
    import torch
    import torch.distributed as dist
    from generativemodels_b200.inferers import LatentDiffusionInferer
    from generativemodels_b200.networks.nets import VQVAE, AutoencoderKL, ControlNet, DiffusionModelUNet
    from generativemodels_b200.networks.schedulers import DDIMScheduler

    def sync():
        torch.cuda.synchronize()

    def maxrank(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    res = {}
    torch.manual_seed(0)
    ae = AutoencoderKL(**C2_AEKL).eval()
    un = redraw_zero_params(DiffusionModelUNet(**C2_UNET).eval(), 2)
    states_out["c2_ae"] = {k: v.clone() for k, v in ae.state_dict().items()}
    states_out["c2_unet"] = {k: v.clone() for k, v in un.state_dict().items()}
    ae, un = ae.cuda(), un.cuda()
    s = DDIMScheduler(**C2_SCHED)
    s.set_timesteps(DDIM_STEPS)
    inf = LatentDiffusionInferer(s, scale_factor=1.0)
    for nb in (1, 32):
        torch.manual_seed(1234 + rank)
        host = torch.randn(nb, 3, 64, 64).pin_memory()
        dev = host.cuda()
        out_host = torch.empty(nb, 1, 256, 256).pin_memory()
        t = maxrank(time_calls(lambda: inf.sample(dev, ae, un, s, verbose=False), 3 if nb == 1 else 2, sync))

        def e2e():
            out_host.copy_(inf.sample(host.cuda(non_blocking=True), ae, un, s, verbose=False), non_blocking=True)
        te = maxrank(time_calls(e2e, 2, sync))
        tf = TF_C2_SAMPLE * nb / t
        res[f"C2_ldm_n{nb}"] = {
            "workload": f"AutoencoderKL (128,128,256) + latent UNet (128,256,512), DDIM-50 + decode, {nb} x 3x64x64 -> "
                        f"1x256x256 per GPU, LatentDiffusionInferer.sample",
            "value": world * nb / t, "unit": "samples/s", "ms_per_call": t * 1e3, "pixels_per_s": world * nb * 65536 / t,
            "algorithmic_tflops": tf, "frac_of_tensor_peak": tf / peak_tf,
            "e2e": {"value": world * nb / te, "unit": "samples/s", "h2d_bytes_per_call": host.numel() * 4 + 4 * DDIM_STEPS,
                    "d2h_bytes_per_call": out_host.numel() * 4}}
    del ae, un
    vq = VQVAE(**C4_VQVAE).eval()
    states_out["c4"] = {k: v.clone() for k, v in vq.state_dict().items()}
    vq = vq.cuda()
    torch.manual_seed(1234 + rank)
    hx = torch.rand(1, 1, 128, 128, 128).pin_memory()
    dx = hx.cuda()
    ho = torch.empty_like(hx).pin_memory()
    t = maxrank(time_calls(lambda: vq(dx), 5, sync))

    def e2e4():
        ho.copy_(vq(hx.cuda(non_blocking=True))[0], non_blocking=True)
    te = maxrank(time_calls(e2e4, 5, sync))
    res["C4_vqvae"] = {"workload": "VQVAE (256,256) 256 codes x 32: encode -> VectorQuantizer -> decode of 1x128^3 per GPU",
                       "value": world * 128 ** 3 / t, "unit": "voxels/s", "ms_per_call": t * 1e3,
                       "algorithmic_tflops": TF_C4_VOLUME / t, "frac_of_tensor_peak": TF_C4_VOLUME / t / peak_tf,
                       "e2e": {"value": world * 128 ** 3 / te, "unit": "voxels/s", "h2d_bytes_per_call": hx.numel() * 4,
                               "d2h_bytes_per_call": ho.numel() * 4}}
    del vq
    u5 = redraw_zero_params(DiffusionModelUNet(out_channels=3, **C5_COMMON).eval(), 3)
    c5 = redraw_zero_params(ControlNet(conditioning_embedding_in_channels=1, conditioning_embedding_num_channels=(16,),
                                       **C5_COMMON).eval(), 4)
    states_out["c5_unet"] = {k: v.clone() for k, v in u5.state_dict().items()}
    states_out["c5_cn"] = {k: v.clone() for k, v in c5.state_dict().items()}
    u5, c5 = u5.cuda(), c5.cuda()
    s5 = DDIMScheduler(num_train_timesteps=1000)
    s5.set_timesteps(DDIM_STEPS)
    mask = c5_mask().cuda()
    torch.manual_seed(1234 + rank)
    h5 = torch.randn(1, 3, 256, 256).pin_memory()
    o5 = torch.empty_like(h5).pin_memory()

    from generativemodels_b200.cuda_graph import graphed

    def cfg_sample(img, unet, cnet, guidance=7.0):
        ctx = torch.cat([-torch.ones(1, 1, 1), torch.ones(1, 1, 1)]).cuda()
        cond = mask.expand(2, -1, -1, -1).contiguous()
        for tt in s5.timesteps:                      # the tutorials' loop (classifier_free_guidance tutorial 304-312)
            x2 = torch.cat([img] * 2)
            ts = torch.Tensor((tt,)).cuda()
            down, mid = cnet(x2, ts, cond, context=ctx)
            eps = unet(x2, ts, context=ctx, down_block_additional_residuals=down, mid_block_additional_residual=mid)
            eu, et = eps.chunk(2)
            img, _ = s5.step(eu + guidance * (et - eu), tt, img)
        return img
    d5 = h5.cuda()
    t_eager = maxrank(time_calls(lambda: cfg_sample(d5, u5, c5), 1, sync))
    # the loop is the user's own (no inferer to replay the networks for them): wrapped once with this package's public
    # CUDA-graph wrapper, as INTEGRATION.md recommends for launch-bound models
    u5g, c5g = graphed(u5), graphed(c5)
    t = maxrank(time_calls(lambda: cfg_sample(d5, u5g, c5g), 1, sync))

    def e2e5():
        o5.copy_(cfg_sample(h5.cuda(non_blocking=True), u5g, c5g), non_blocking=True)
    te = maxrank(time_calls(e2e5, 1, sync))
    tf = TF_C5_STEP * DDIM_STEPS / t
    res["C5_controlnet_cfg"] = {
        "workload": "ControlNet + conditioned UNet (128,256,256) at 3x256x256, classifier-free guidance 7 (batch doubled "
                    "inside the step), DDIM-50, one guided sample per GPU, public nn.Module / scheduler API",
        "value": world / t, "unit": "guided samples/s", "ms_per_call": t * 1e3, "values_per_s": world * 3 * 65536 / t,
        "ms_per_call_eager": t_eager * 1e3, "networks": "cuda_graph.graphed(unet), graphed(controlnet)",
        "algorithmic_tflops": tf, "frac_of_tensor_peak": tf / peak_tf,
        "e2e": {"value": world / te, "unit": "guided samples/s", "h2d_bytes_per_call": h5.numel() * 4 + 4 * DDIM_STEPS,
                "d2h_bytes_per_call": o5.numel() * 4}}
    del u5, c5, u5g, c5g
    torch.cuda.empty_cache()
    return res


def run_b200(args):
    import torch
    import torch.distributed as dist

    from generativemodels_b200 import _lib, ops
    from generativemodels_b200.inferers import DiffusionInferer
    from generativemodels_b200.networks.schedulers import DDIMScheduler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.require_device()
    peak_tf, peak_gbs, which = peaks()

    model = build_model_state()
    c3_state = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.cuda()
    vol = tuple(args.volume) if args.volume else C3_VOLUME
    voxels = vol[0] * vol[1] * vol[2] * args.batch
    sched = DDIMScheduler(**C3_SCHED)
    sched.set_timesteps(DDIM_STEPS)
    torch.manual_seed(1234)
    noise_all = torch.randn(world * args.batch, 1, *vol)            # one global draw, sliced per rank (SURVEY section 8e)
    noise_host = noise_all[rank * args.batch:(rank + 1) * args.batch].contiguous().pin_memory()
    x = noise_host.cuda(non_blocking=True)
    inst = Instrument(lib, ops, _lib)

    def one_step(x, t):
        eps = model(x, timesteps=torch.Tensor((t,)).to(x.device))
        x, _ = sched.step(eps, t, x)
        return x

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    ts = [int(t) for t in sched.timesteps]
    k = 0
    for _ in range(args.warmup):
        x = one_step(x, ts[k % DDIM_STEPS]); k += 1
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    inst.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        x = one_step(x, ts[k % DDIM_STEPS]); k += 1
    if world > 1:                                   # the path's only collective: gather the finished samples
        gathered = [torch.empty_like(x) for _ in range(world)]
        dist.all_gather(gathered, x)
    e1.record()
    barrier()
    inst.stop()
    ms_local = e0.elapsed_time(e1)
    dumped = {"sample": x.cpu()} if args.dump_outputs and rank == 0 else None     # what this rank's last step returned
    clock_line = clocks.stop() if rank == 0 else None
    ms_total, per_rank = ms_local, [ms_local / args.steps]
    if world > 1:
        allms = [torch.zeros(1, device="cuda") for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms_local], device="cuda"))
        per_rank = [float(t.item()) / args.steps for t in allms]
        ms_total = max(per_rank) * args.steps
    ms_step = ms_total / args.steps
    value = world * voxels / (DDIM_STEPS * ms_step * 1e-3)
    n_launch = inst.n
    finite = bool(torch.isfinite(x).all())
    times = {key: inst.ms(key) for key in inst.ev}
    work = dict(inst.work)
    counts = {key: len(v) for key, v in inst.ev.items()}

    # ---- e2e through the public API: pinned host noise in, pinned host result out, the gather included ----
    ke = args.steps
    sched_e = DDIMScheduler(**C3_SCHED)
    sched_e.set_timesteps(ke)
    inferer = DiffusionInferer(sched_e)
    out_host = torch.empty_like(noise_host).pin_memory()
    barrier()
    t0 = time.perf_counter()
    xin = noise_host.cuda(non_blocking=True)
    sample = inferer.sample(input_noise=xin, diffusion_model=model, scheduler=sched_e, verbose=False)
    if world > 1:
        gathered = [torch.empty_like(sample) for _ in range(world)]
        dist.all_gather(gathered, sample)
    out_host.copy_(sample, non_blocking=True)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax.item())
    e2e_value = world * voxels / (e2e_s * DDIM_STEPS / ke)
    nbytes = noise_host.numel() * 4
    del model, x, sample
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations ----
    states, others = {}, None
    if not args.no_other_configs:
        others = other_configs_gpu(world, rank, peak_tf, states)

    if rank == 0:
        cpu_line = None
        if world == 1 and not args.no_cpu_baseline:
            v, sec, cores, kind = cpu_c3_steps(c3_state, 5, 1)
            cpu_line = {"value": v, "unit": "voxels/s", "cores": cores, "kind": kind,
                        "sample": f"{'the unmodified reference (oracle/_ref)' if kind == 'reference' else 'oracle port'}: "
                                  f"UNet forward + DDIM step on 1x1x{'x'.join(map(str, CPU_VOLUME))}, 5 steps after 1 "
                                  f"warm-up ({sec:.2f} s/step), {cores} threads"}
            if others is not None:
                for key, leg in cpu_other_configs(states).items():
                    others[key]["cpu_baseline"] = leg
        achieved = work["conv"] / (times["conv"] * 1e-3) / 1e12 if times["conv"] > 0 else 0.0
        secondary = []
        if times["attn"] > 0:
            a = work["attn"] / (times["attn"] * 1e-3) / 1e12
            secondary.append({"kernel": "flash_attn_kernel (self-attention T = S = 89 600, head 512)", "bound": "tensor",
                              "achieved": a, "peak": peak_tf, "unit": "TFLOP/s", "frac": a / peak_tf,
                              "share_of_step": times["attn"] / ms_local, "launches_timed": counts["attn"]})
        for key, label in (("gn_apply", "gn_apply_kernel (GroupNorm apply + SiLU: 1 read + 1 write, 16-bit)"),
                           ("ddim", "ddim_step_kernel (2 reads + 2 writes, fp32)")):
            if times[key] > 0:
                g = work[key] / (times[key] * 1e-3) / 1e9
                secondary.append({"kernel": label, "bound": "hbm", "achieved": g, "peak": peak_gbs, "unit": "GB/s",
                                  "frac": g / peak_gbs, "share_of_step": times[key] / ms_local,
                                  "launches_timed": counts[key]})
        line = {
            "metric": METRIC, "value": value, "unit": "voxels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": _lib.ACT_DTYPE, "data": "synthetic",
            "config": {"workload": "C3: 3D DiffusionModelUNet (256,256,512) attn (F,F,T) heads (0,0,512), DDIM-50; "
                                   "one step = UNet forward + DDIMScheduler.step",
                       "volume": list(vol), "per_gpu_batch": args.batch, "samples_per_s": value / (voxels / args.batch),
                       "operands": f"{_lib.ACT_DTYPE} x {_lib.ACT_DTYPE} -> fp32 accumulate (tcgen05 kind::f16)",
                       "l2": "per-step working set (tens of GB of activations) >> 126 MB L2; no explicit flush",
                       "finite_output": finite, "ms_per_step_per_rank": per_rank,
                       "algorithmic_tflop_per_forward": TF_C3_FORWARD,
                       "whole_step_tflops": TF_C3_FORWARD * (voxels / (C3_VOLUME[0] * C3_VOLUME[1] * C3_VOLUME[2]))
                                            / (ms_step * 1e-3)},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved / peak_tf if peak_tf else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel (the 256->256
                         # 3x3x3 conv at 160x224x160; algorithmic 5.88e9 B) from the ncu --set full capture
                         # profiles/r2_ncu_igemm_pair_conv256_fullres_final3_details.txt at the round's last commit
                         # (4.33 GB read + 2.91 GB written, tensor pipe 99.5 % of active cycles, 13.02 ms at 1.31 GHz;
                         # the capture earlier in the round, r2_ncu_igemm_pair_conv256_fullres_details.txt: 6.37e9)
                         "traffic": 7.24e9,
                         "kernel": "igemm_tc_kernel<256,6,pair> (3x3x3 convolutions, tcgen05 cta_group::2)",
                         "peak_source": which + " sustained 16-bit GEMM",
                         "share_of_step": times["conv"] / ms_local if ms_local else None,
                         "launches_timed": counts["conv"], "secondary": secondary},
            "cpu_baseline": cpu_line,
            "e2e": {"value": e2e_value, "unit": "voxels/s", "h2d_bytes_per_step": nbytes / ke + 4,
                    "d2h_bytes_per_step": nbytes / ke, "steps_run": ke, "includes_all_gather": world > 1,
                    "api": "DiffusionInferer.sample(pinned host noise -> cuda, DDIMScheduler) -> pinned host"},
            "gpu_launches": n_launch,
            "clocks": clock_line,
            "other_configs": others,
        }
        print(json.dumps(line))
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="samples per GPU")
    ap.add_argument("--volume", type=int, nargs=3, default=None, help="override the C3 volume (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
