"""Pin oracle/torch_oracle.py against the UNMODIFIED reference through stored vectors.

tests/golden/g_oracle_vs_reference.pt holds what the reference computed for every case below, on CPU fp32
(tests/golden/make_golden_oracle_vs_reference.py).  Weights come from tests.golden.configs.recipe_state_dict, drawn here
on this package's modules and there on the reference's (same keys and shapes); inputs come from the seeded helpers
below, which the generator shares."""
import hashlib
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import torch_oracle as O
from tests.golden import configs as G

GOLD = Path(__file__).resolve().parent / "golden" / "g_oracle_vs_reference.pt"
CN_SEEDS = (2024, 2025)          # recipe seeds of the ControlNet and of the UNet it feeds
# recipe seeds of the VQVAE and of the transformer of the greedy sampler; with 2025 the transformer's top token is the
# BOS token at some step, which the reference removes after its top-k cut and then cannot sample from
GREEDY_SEEDS = (2024, 2026)


@pytest.fixture(scope="module")
def ref():
    """The reference's outputs, per case."""
    return torch.load(GOLD, weights_only=False)


def recipe(cls, seed=2024, **kw):
    """Recipe weights of a module of class ``cls`` built by this package (keys and shapes only)."""
    from generativemodels_b200.networks import nets
    return G.recipe_state_dict(getattr(nets, cls)(**kw), seed)


def digest(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def sample(t, n=1024):
    """A fixed, seeded sample of ``n`` elements of ``t``: what is stored of the larger reference outputs."""
    idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n]
    return t.reshape(-1)[idx]


def _close(a, b, tol=2e-5):
    err = (a - b).abs().max().item()
    assert err <= tol * max(1.0, b.abs().max().item()), f"max abs err {err:.3e}"


# seeded inputs, shared with the generator
def unet_inputs(name):
    inp = G.UNET_INPUTS[name]
    torch.manual_seed(1)
    x = torch.randn(inp["shape"])
    t = torch.randint(0, 1000, (inp["shape"][0],)).long()
    ctx = torch.randn(inp["context"]) if "context" in inp else None
    cls = torch.randint(0, 5, (inp["shape"][0],)) if inp.get("classes") else None
    return x, t, ctx, cls


def controlnet_inputs():
    torch.manual_seed(2)
    x, cond, ctx = torch.randn(2, 3, 16, 16), torch.rand(2, 1, 16, 16), torch.randn(2, 1, 8)
    return x, torch.tensor([10, 500]).long(), cond, ctx


def controlnet_unet_kwargs():
    kw = {k: v for k, v in G.CONTROLNET_CASE.items() if not k.startswith("conditioning_embedding")}
    return dict(out_channels=3, **kw)


def aekl_input(name):
    torch.manual_seed(3)
    return torch.randn(G.AEKL_INPUTS[name])


def vqvae_input(name):
    torch.manual_seed(4)
    return torch.rand(G.VQVAE_INPUTS[name])


def scheduler_start():
    torch.manual_seed(5)
    return torch.randn(2, 3, 8, 8)


def scheduler_model_output(x, t):
    """Deterministic stand-in for the network; rational rather than transcendental, so that it rounds the same on
    every CPU and the stored trajectory can be compared bit for bit."""
    return x * 0.7 / (1.0 + x.abs()) + 0.01 * float(t)


def inferer_noise():
    torch.manual_seed(7)
    return torch.randn(1, 1, 16, 16)


def likelihood_inputs():
    torch.manual_seed(5)
    x = torch.rand(2, 1, 16, 16) * 2 - 1
    x[0, 0, 0, :4] = torch.tensor([-1.0, 1.0, -0.9995, 0.9995])          # both edge bins of the discretised decoder
    return x, torch.randn(2, 1, 16, 16)


def spade_unet_inputs(name):
    inp = G.SPADE_UNET_INPUTS[name]
    torch.manual_seed(1)
    x = torch.randn(*inp["shape"])
    t = torch.randint(0, 1000, (inp["shape"][0],)).long()
    ctx = torch.randn(*inp["context"]) if "context" in inp else None
    return x, t, G.seg_onehot(inp["seg"]), ctx


def spade_aekl_inputs(name):
    torch.manual_seed(1)
    x = torch.randn(*G.SPADE_AEKL_INPUTS[name])
    return x, G.seg_onehot((x.shape[0], G.SPADE_AEKL_CASES[name]["label_nc"], *x.shape[2:]))


def transformer_kwargs(cross):
    return dict(num_tokens=11, max_seq_len=16, attn_layers_dim=32, attn_layers_depth=2, attn_layers_heads=4,
                with_cross_attention=cross)


def transformer_inputs(cross):
    torch.manual_seed(6)
    x = torch.randint(0, 11, (2, 9))
    return x, (torch.randn(2, 3, 32) if cross else None)


def greedy_transformer_kwargs():
    return dict(num_tokens=G.VQVAE_CASES["vqvae2d"]["num_embeddings"] + 1, max_seq_len=10, attn_layers_dim=32,
                attn_layers_depth=2, attn_layers_heads=4)


ORDERINGS = (
    dict(ordering_type="s_curve", spatial_dims=2, dimensions=(1, 3, 4), reflected_spatial_dims=(True, False)),
    dict(ordering_type="raster_scan", spatial_dims=3, dimensions=(1, 2, 3, 4), transpositions_axes=((2, 0, 1),),
         rot90_axes=((0, 1),), reflected_spatial_dims=(False, True, True)),
    dict(ordering_type="s_curve", spatial_dims=3, dimensions=(1, 3, 2, 4),
         transformation_order=("reflect", "transpose", "rotate_90"),
         reflected_spatial_dims=(True, True, False), transpositions_axes=((1, 0, 2),)),
)


def pndm_restart_inputs():
    torch.manual_seed(0)
    x = torch.randn(1, 1, 8, 8)
    return x, [torch.randn(1, 1, 8, 8) for _ in range(8)]


def pndm_drive(s, x, outs):
    """Abort a loop mid-Runge-Kutta cycle, restart on the same scheduler and run 8 steps."""
    s.set_timesteps(4)
    y = x
    for t, e in zip(s.timesteps[:2], outs):
        y, _ = s.step(e.clone(), int(t), y)
    s.set_timesteps(4)
    y = x
    for t, e in zip(s.timesteps[:8], outs):
        y, _ = s.step(e.clone(), int(t), y)
    return y


@pytest.mark.parametrize("name", list(G.UNET_CASES))
def test_unet(ref, name):
    kw = G.UNET_CASES[name]
    x, t, ctx, cls = unet_inputs(name)
    with torch.no_grad():
        got = O.unet_forward(recipe("DiffusionModelUNet", **kw), G.unet_oracle_cfg(kw), x, t, context=ctx,
                             class_labels=cls)
    _close(got, ref["unet"][name])


def test_controlnet(ref):
    kw, want = G.CONTROLNET_CASE, ref["controlnet"]
    csd = recipe("ControlNet", CN_SEEDS[0], **kw)
    usd = recipe("DiffusionModelUNet", CN_SEEDS[1], **controlnet_unet_kwargs())
    x, t, cond, ctx = controlnet_inputs()
    cfg = G.unet_oracle_cfg(kw)
    with torch.no_grad():
        d_g, m_g = O.controlnet_forward(csd, cfg, x, t, cond, 0.7, ctx)
        assert [tuple(a.shape) for a in d_g] == want["down_shapes"] and tuple(m_g.shape) == want["mid_shape"]
        for a, b in zip(d_g, want["down"]):
            _close(sample(a), b)
        _close(sample(m_g), want["mid"])
        got = O.unet_forward(usd, cfg, x, t, context=ctx, down_block_additional_residuals=d_g,
                             mid_block_additional_residual=m_g)
    _close(got, want["y"])


@pytest.mark.parametrize("name", list(G.AEKL_CASES))
def test_autoencoderkl(ref, name):
    kw, want = G.AEKL_CASES[name], ref["autoencoderkl"][name]
    sd, cfg = recipe("AutoencoderKL", **kw), G.aekl_oracle_cfg(kw)
    x = aekl_input(name)
    with torch.no_grad():
        mu_g, sig_g = O.autoencoderkl_encode(sd, cfg, x)
        _close(mu_g, want["mu"])
        _close(sig_g, want["sigma"])
        _close(O.autoencoderkl_decode(sd, cfg, want["mu"]), want["rec"])


@pytest.mark.parametrize("name", list(G.VQVAE_CASES))
def test_vqvae(ref, name):
    kw, want = G.VQVAE_CASES[name], ref["vqvae"][name]
    sd, cfg = recipe("VQVAE", **kw), G.vqvae_oracle_cfg(kw)
    cb = sd["quantizer.quantizer.embedding.weight"]
    x = vqvae_input(name)
    with torch.no_grad():
        rec_g, loss_g, idx_g = O.vqvae_forward(sd, cfg, x)
        assert torch.equal(idx_g, want["idx"])
        _close(rec_g, want["rec"])
        _close(loss_g, want["loss"])
        _close(O.vqvae_decode(sd, cfg, O.vq_embed(cb, want["idx"])), want["dec"])
        _close(O.vq_forward(cb, want["z"])[3], want["perplexity"])


SCHED = [
    ("ddim", dict(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0015, beta_end=0.0195), 50),
    ("ddim", dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0005, beta_end=0.0195,
                  clip_sample=False), 50),
    ("ddim", dict(num_train_timesteps=100, prediction_type="v_prediction", set_alpha_to_one=False, steps_offset=1), 10),
    # (cosine has alphas_cumprod[0] == 1 exactly: t = 0 divides by zero in the reference itself, so offset by 1)
    ("ddim", dict(num_train_timesteps=100, prediction_type="sample", schedule="cosine", steps_offset=1,
                  set_alpha_to_one=False), 7),
    ("ddpm", dict(num_train_timesteps=1000), 4),
    ("ddpm", dict(num_train_timesteps=100, variance_type="fixed_large", prediction_type="v_prediction",
                  schedule="sigmoid_beta"), 10),
    ("pndm", dict(num_train_timesteps=1000, skip_prk_steps=True), 20),
    ("pndm", dict(num_train_timesteps=1000, skip_prk_steps=False), 20),
    ("pndm", dict(num_train_timesteps=100, skip_prk_steps=False, prediction_type="v_prediction",
                  set_alpha_to_one=True, steps_offset=1), 10),
]


def scheduler_trajectory(s, kind):
    """Run the stand-in model output through scheduler ``s`` (timesteps set): digest of every step's sample, and the
    last sample."""
    x = scheduler_start()
    digests = []
    for t in s.timesteps:
        eps = scheduler_model_output(x, t)
        if kind == "ddpm":
            x, _ = s.step(eps, int(t), x, generator=torch.Generator().manual_seed(int(t)))
        else:
            x, _ = s.step(eps, int(t), x)
        digests.append(digest(x))
    return digests, x


@pytest.mark.parametrize("i", range(len(SCHED)), ids=[f"{k}-{i}" for i, (k, _, _) in enumerate(SCHED)])
def test_scheduler_trajectory(ref, i):
    """Identical model-output sequence through the reference scheduler and the restated one: every step equal."""
    kind, kw, steps = SCHED[i]
    want = ref["scheduler"][i]
    M = {"ddim": O.DDIMOracle, "ddpm": O.DDPMOracle, "pndm": O.PNDMOracle}[kind](**kw)
    M.set_timesteps(steps)
    assert torch.equal(M.timesteps, want["timesteps"])
    assert digest(M.alphas_cumprod) == want["alphas_cumprod"]
    digests, x = scheduler_trajectory(M, kind)
    assert len(digests) == len(want["digests"])
    for t, a, b in zip(M.timesteps, digests, want["digests"]):
        assert a == b, f"diverged at t={int(t)}"
    assert torch.equal(x, want["sample"])


def test_inferer_sample(ref):
    kw = G.UNET_CASES["unet2d_attn"]
    skw = dict(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0015, beta_end=0.0195)
    M = O.DDIMOracle(**skw)
    M.set_timesteps(5)
    cfg, sd = G.unet_oracle_cfg(kw), recipe("DiffusionModelUNet", **kw)
    with torch.no_grad():
        got = O.diffusion_sample(lambda x, t, c: O.unet_forward(sd, cfg, x, t, context=c), M, inferer_noise())
    _close(got, ref["inferer_sample"], 1e-4)


@pytest.mark.parametrize("ptype,clip", [("epsilon", True), ("v_prediction", False), ("sample", True)])
def test_get_likelihood(ref, ptype, clip):
    """Oracle get_likelihood vs the reference's DiffusionInferer.get_likelihood (inferer.py:145-277), same noise."""
    kw = G.UNET_CASES["unet2d_attn"]
    M = O.DDPMOracle(num_train_timesteps=12, prediction_type=ptype, clip_sample=clip)
    M.set_timesteps(12)
    x, noise = likelihood_inputs()
    cfg, sd = G.unet_oracle_cfg(kw), recipe("DiffusionModelUNet", **kw)
    with torch.no_grad():
        got = O.get_likelihood(lambda xx, t, c: O.unet_forward(sd, cfg, xx, t, context=c), M, x, noise)
    _close(got, ref["likelihood"][ptype], 1e-4)


@pytest.mark.parametrize("name", list(G.SPADE_UNET_CASES))
def test_spade_unet(ref, name):
    """SPADEDiffusionModelUNet (spade_diffusion_model_unet.py:612-912): SPADE norms in the up path, incl. the
    InstanceNorm that monai's Convolution puts on mlp_gamma / mlp_beta."""
    kw = G.SPADE_UNET_CASES[name]
    x, t, seg, ctx = spade_unet_inputs(name)
    with torch.no_grad():
        got = O.unet_forward(recipe("SPADEDiffusionModelUNet", **kw), G.unet_oracle_cfg(kw), x, t, context=ctx, seg=seg)
    _close(got, ref["spade_unet"][name])


@pytest.mark.parametrize("name", list(G.SPADE_AEKL_CASES))
def test_spade_autoencoderkl(ref, name):
    """SPADEAutoencoderKL.encode / decode(z, seg) (spade_autoencoderkl.py:425-469)."""
    kw, want = G.SPADE_AEKL_CASES[name], ref["spade_autoencoderkl"][name]
    sd, cfg = recipe("SPADEAutoencoderKL", **kw), G.aekl_oracle_cfg(kw)
    x, seg = spade_aekl_inputs(name)
    with torch.no_grad():
        gmu, gsigma = O.autoencoderkl_encode(sd, cfg, x)
        grec = O.autoencoderkl_decode(sd, cfg, gmu, seg=seg)
    _close(gmu, want["mu"])
    _close(gsigma, want["sigma"])
    _close(grec, want["rec"])


def test_ordering(ref):
    """utils/ordering.py: raster / s-curve scans of transposed, rotated and reflected index grids."""
    assert len(ref["ordering"]) == len(ORDERINGS)
    for kw, want in zip(ORDERINGS, ref["ordering"]):
        assert np.array_equal(want, O.sequence_ordering(**kw))


@pytest.mark.parametrize("cross", [False, True])
def test_transformer(ref, cross):
    """DecoderOnlyTransformer.forward (nets/transformer.py:96-106)."""
    sd = recipe("DecoderOnlyTransformer", **transformer_kwargs(cross))
    x, ctx = transformer_inputs(cross)
    with torch.no_grad():
        _close(O.transformer_forward(sd, 4, x, ctx), ref["transformer"][cross])


def test_transformer_greedy_sampling(ref):
    """VQVAETransformerInferer.sample with top_k = 1 (inferer.py:1183-1245) against the oracle's greedy loop, incl.
    the sliding window once the sequence outgrows max_seq_len."""
    vkw = G.VQVAE_CASES["vqvae2d"]
    vsd = recipe("VQVAE", GREEDY_SEEDS[0], **vkw)
    tsd = recipe("DecoderOnlyTransformer", GREEDY_SEEDS[1], **greedy_transformer_kwargs())
    K = vkw["num_embeddings"]
    order = O.sequence_ordering("raster_scan", 2, (1, 4, 4))
    with torch.no_grad():
        seq = O.transformer_sample_greedy(tsd, 4, 10, K, 16, 2)
        seq = seq[:, torch.argsort(torch.as_tensor(order))].reshape(2, 4, 4)
        emb = O.vq_embed(vsd["quantizer.quantizer.embedding.weight"], seq)
        got = O.vqvae_decode(vsd, G.vqvae_oracle_cfg(vkw), emb)
    _close(got, ref["greedy_sample"])


def test_pndm_restart_mid_runge_kutta(ref):
    """The reference keeps a stale Runge-Kutta accumulator when a loop is aborted mid-cycle and restarted on the same
    scheduler (``+=`` at phase 0, pndm.py:208; set_timesteps resets ets / counter only): the oracle follows it."""
    want = ref["pndm_restart"]
    assert not torch.allclose(want["restarted"], want["fresh"])     # the stale sum really is inherited by the reference
    got = pndm_drive(O.PNDMOracle(num_train_timesteps=1000, skip_prk_steps=False), *pndm_restart_inputs())
    _close(got, want["restarted"], 1e-6)
