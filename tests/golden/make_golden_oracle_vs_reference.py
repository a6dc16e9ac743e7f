"""Generate tests/golden/g_oracle_vs_reference.pt by running the UNMODIFIED reference (CPU fp32, MONAI shim) on the
cases of tests/test_oracle_vs_reference.py:   python -m tests.golden.make_golden_oracle_vs_reference

Weights come from tests.golden.configs.recipe_state_dict and inputs from the test module's seeded helpers, so the
fixture holds only what the reference computed."""
from pathlib import Path

import torch

from tests import test_oracle_vs_reference as T    # before the reference import: it has its own `tests` package
from tests.golden import configs as G
from oracle import ref_import

OUT = Path(__file__).resolve().parent / "g_oracle_vs_reference.pt"


def main():
    ref_import.import_reference()
    import generative.networks.nets as nets
    import generative.networks.schedulers as sch
    from generative.inferers import DiffusionInferer, VQVAETransformerInferer
    from generative.utils.ordering import Ordering

    def model(cls, seed=2024, **kw):
        m = getattr(nets, cls)(**kw).eval()
        G.recipe_state_dict(m, seed)
        return m

    torch.set_grad_enabled(False)
    fx = {}
    fx["unet"] = {}
    for name, kw in G.UNET_CASES.items():
        x, t, ctx, cls = T.unet_inputs(name)
        fx["unet"][name] = model("DiffusionModelUNet", **kw)(x, t, context=ctx, class_labels=cls)

    cn = model("ControlNet", T.CN_SEEDS[0], **G.CONTROLNET_CASE)
    un = model("DiffusionModelUNet", T.CN_SEEDS[1], **T.controlnet_unet_kwargs())
    x, t, cond, ctx = T.controlnet_inputs()
    down, mid = cn(x, t, cond, conditioning_scale=0.7, context=ctx)
    y = un(x, t, context=ctx, down_block_additional_residuals=down, mid_block_additional_residual=mid)
    fx["controlnet"] = dict(down=[T.sample(d) for d in down], down_shapes=[tuple(d.shape) for d in down],
                            mid=T.sample(mid), mid_shape=tuple(mid.shape), y=y)

    fx["autoencoderkl"] = {}
    for name, kw in G.AEKL_CASES.items():
        m = model("AutoencoderKL", **kw)
        mu, sigma = m.encode(T.aekl_input(name))
        fx["autoencoderkl"][name] = dict(mu=mu, sigma=sigma, rec=m.decode(mu))

    fx["vqvae"] = {}
    for name, kw in G.VQVAE_CASES.items():
        m = model("VQVAE", **kw)
        x = T.vqvae_input(name)
        rec, loss = m(x)
        idx = m.index_quantize(x)
        z = m.encode(x)
        fx["vqvae"][name] = dict(rec=rec, loss=loss, idx=idx, dec=m.decode_samples(idx), z=z,
                                 perplexity=m.quantizer.perplexity.clone())

    fx["scheduler"] = []
    for kind, kw, steps in T.SCHED:
        s = {"ddim": sch.DDIMScheduler, "ddpm": sch.DDPMScheduler, "pndm": sch.PNDMScheduler}[kind](**kw)
        s.set_timesteps(steps)
        timesteps, alphas_cumprod = s.timesteps.clone(), T.digest(s.alphas_cumprod)
        digests, x = T.scheduler_trajectory(s, kind)
        fx["scheduler"].append(dict(timesteps=timesteps, alphas_cumprod=alphas_cumprod, digests=digests, sample=x))

    kw = G.UNET_CASES["unet2d_attn"]
    m = model("DiffusionModelUNet", **kw)
    s = sch.DDIMScheduler(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0015, beta_end=0.0195)
    s.set_timesteps(5)
    fx["inferer_sample"] = DiffusionInferer(s).sample(input_noise=T.inferer_noise(), diffusion_model=m, scheduler=s,
                                                      verbose=False)
    fx["likelihood"] = {}
    randn_like = torch.randn_like
    try:
        for ptype, clip in (("epsilon", True), ("v_prediction", False), ("sample", True)):
            s = sch.DDPMScheduler(num_train_timesteps=12, prediction_type=ptype, clip_sample=clip)
            s.set_timesteps(12)
            x, noise = T.likelihood_inputs()
            torch.randn_like = lambda t: noise.clone()       # the reference draws its noise inside get_likelihood
            fx["likelihood"][ptype] = DiffusionInferer(s).get_likelihood(inputs=x, diffusion_model=m, scheduler=s,
                                                                         verbose=False)
    finally:
        torch.randn_like = randn_like

    fx["spade_unet"] = {}
    for name, kw in G.SPADE_UNET_CASES.items():
        x, t, seg, ctx = T.spade_unet_inputs(name)
        fx["spade_unet"][name] = model("SPADEDiffusionModelUNet", **kw)(x, t, seg, context=ctx)
    fx["spade_autoencoderkl"] = {}
    for name, kw in G.SPADE_AEKL_CASES.items():
        m = model("SPADEAutoencoderKL", **kw)
        x, seg = T.spade_aekl_inputs(name)
        mu, sigma = m.encode(x)
        fx["spade_autoencoderkl"][name] = dict(mu=mu, sigma=sigma, rec=m.decode(mu, seg))

    fx["ordering"] = [Ordering(**kw).get_sequence_ordering() for kw in T.ORDERINGS]

    fx["transformer"] = {}
    for cross in (False, True):
        x, ctx = T.transformer_inputs(cross)
        fx["transformer"][cross] = model("DecoderOnlyTransformer", **T.transformer_kwargs(cross))(x, context=ctx)

    vq = model("VQVAE", T.GREEDY_SEEDS[0], **G.VQVAE_CASES["vqvae2d"])
    tr = model("DecoderOnlyTransformer", T.GREEDY_SEEDS[1], **T.greedy_transformer_kwargs())
    start = torch.full((2, 1), G.VQVAE_CASES["vqvae2d"]["num_embeddings"])
    fx["greedy_sample"] = VQVAETransformerInferer().sample((4, 4), start, vq, tr, Ordering("raster_scan", 2, (1, 4, 4)),
                                                           top_k=1, verbose=False)

    x, outs = T.pndm_restart_inputs()
    restarted = T.pndm_drive(sch.PNDMScheduler(num_train_timesteps=1000, skip_prk_steps=False), x, outs)
    fresh = sch.PNDMScheduler(num_train_timesteps=1000, skip_prk_steps=False)
    fresh.set_timesteps(4)
    y = x
    for t, e in zip(fresh.timesteps[:8], outs):
        y, _ = fresh.step(e.clone(), int(t), y)
    fx["pndm_restart"] = dict(restarted=restarted, fresh=y)

    torch.save(fx, OUT)
    print(OUT.name, OUT.stat().st_size)


if __name__ == "__main__":
    main()
