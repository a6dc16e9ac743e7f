"""Small model configurations shared by the golden-vector generator and the parity tests.

Each entry: constructor kwargs in the reference's own vocabulary + the oracle cfg derived from them.  Channels are
multiples of 8 (and of the group count) so the CUDA path runs its vectorised kernels; sizes are chosen so the CPU
oracle finishes in well under a second per forward.
"""

UNET_CASES = {
    "unet2d_attn": dict(spatial_dims=2, in_channels=1, out_channels=1, num_res_blocks=1, num_channels=(32, 64, 64),
                        attention_levels=(False, True, True), norm_num_groups=8, num_head_channels=(0, 32, 64)),
    "unet3d_attn": dict(spatial_dims=3, in_channels=1, out_channels=1, num_res_blocks=(1, 2), num_channels=(32, 64),
                        attention_levels=(False, True), norm_num_groups=8, num_head_channels=(0, 64)),
    "unet2d_small_heads": dict(spatial_dims=2, in_channels=3, out_channels=3, num_res_blocks=1, num_channels=(16, 16),
                               attention_levels=(True, True), norm_num_groups=8, num_head_channels=4),
    "unet2d_cross": dict(spatial_dims=2, in_channels=3, out_channels=3, num_res_blocks=1, num_channels=(32, 64),
                         attention_levels=(False, True), norm_num_groups=8, num_head_channels=(0, 32),
                         with_conditioning=True, cross_attention_dim=8, transformer_num_layers=1),
    "unet2d_updown_class": dict(spatial_dims=2, in_channels=2, out_channels=2, num_res_blocks=1, num_channels=(16, 32),
                                attention_levels=(False, True), norm_num_groups=8, num_head_channels=16,
                                resblock_updown=True, num_class_embeds=5),
}
UNET_INPUTS = {
    "unet2d_attn": dict(shape=(2, 1, 16, 16)),
    "unet3d_attn": dict(shape=(1, 1, 8, 12, 8)),
    "unet2d_small_heads": dict(shape=(2, 3, 8, 8)),
    "unet2d_cross": dict(shape=(2, 3, 16, 16), context=(2, 3, 8)),
    "unet2d_updown_class": dict(shape=(2, 2, 16, 16), classes=True),
}

CONTROLNET_CASE = dict(spatial_dims=2, in_channels=3, num_res_blocks=1, num_channels=(32, 64),
                       attention_levels=(False, True), norm_num_groups=8, num_head_channels=(0, 32),
                       with_conditioning=True, cross_attention_dim=8, conditioning_embedding_in_channels=1,
                       conditioning_embedding_num_channels=(16,))

AEKL_CASES = {
    "aekl2d": dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(16, 32), latent_channels=3,
                   num_res_blocks=(1, 1), norm_num_groups=8, attention_levels=(False, False),
                   with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False),
    "aekl3d_attn": dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(16, 16), latent_channels=4,
                        num_res_blocks=(1, 1), norm_num_groups=8, attention_levels=(False, True),
                        with_encoder_nonlocal_attn=True, with_decoder_nonlocal_attn=True),
    "aekl2d_convT": dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(16, 32), latent_channels=3,
                         num_res_blocks=(1, 1), norm_num_groups=8, attention_levels=(False, False),
                         with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False, use_convtranspose=True),
}
AEKL_INPUTS = {"aekl2d": (2, 1, 16, 16), "aekl3d_attn": (1, 1, 8, 8, 8), "aekl2d_convT": (1, 1, 16, 16)}

VQVAE_CASES = {
    "vqvae3d": dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(16, 16), num_res_channels=16,
                    num_res_layers=1, downsample_parameters=((2, 4, 1, 1),) * 2,
                    upsample_parameters=((2, 4, 1, 1, 0),) * 2, num_embeddings=32, embedding_dim=8),
    "vqvae2d": dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(16, 32), num_res_channels=(16, 32),
                    num_res_layers=2, downsample_parameters=((2, 4, 1, 1),) * 2,
                    upsample_parameters=((2, 4, 1, 1, 0),) * 2, num_embeddings=64, embedding_dim=16),
}
VQVAE_INPUTS = {"vqvae3d": (1, 1, 16, 16, 16), "vqvae2d": (2, 1, 32, 32)}


SPADE_UNET_CASES = {
    "spade_unet2d": dict(spatial_dims=2, in_channels=1, out_channels=1, label_nc=3, num_res_blocks=1,
                         num_channels=(32, 64), attention_levels=(False, True), norm_num_groups=8,
                         num_head_channels=(0, 32), spade_intermediate_channels=16),
    "spade_unet3d_updown": dict(spatial_dims=3, in_channels=2, out_channels=2, label_nc=4, num_res_blocks=(1, 2),
                                num_channels=(16, 16), attention_levels=(False, False), norm_num_groups=8,
                                resblock_updown=True, spade_intermediate_channels=8),
    "spade_unet2d_cross": dict(spatial_dims=2, in_channels=1, out_channels=1, label_nc=3, num_res_blocks=1,
                               num_channels=(16, 32), attention_levels=(False, True), norm_num_groups=8,
                               num_head_channels=(0, 16), with_conditioning=True, cross_attention_dim=8,
                               transformer_num_layers=1),
}
SPADE_UNET_INPUTS = {"spade_unet2d": dict(shape=(2, 1, 16, 16), seg=(2, 3, 32, 32)),
                     "spade_unet3d_updown": dict(shape=(1, 2, 8, 8, 8), seg=(1, 4, 8, 8, 8)),
                     "spade_unet2d_cross": dict(shape=(2, 1, 16, 16), seg=(2, 3, 16, 16), context=(2, 3, 8))}
SPADE_AEKL_CASES = {
    "spade_aekl2d": dict(spatial_dims=2, label_nc=3, in_channels=1, out_channels=1, num_channels=(16, 16, 32),
                         latent_channels=4, attention_levels=(False, False, True), num_res_blocks=1, norm_num_groups=8,
                         spade_intermediate_channels=8),
    "spade_aekl3d": dict(spatial_dims=3, label_nc=2, in_channels=1, out_channels=1, num_channels=(16, 16),
                         latent_channels=3, attention_levels=(False, False), num_res_blocks=(1, 2), norm_num_groups=8,
                         with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False,
                         spade_intermediate_channels=8),
}
SPADE_AEKL_INPUTS = {"spade_aekl2d": (2, 1, 16, 16), "spade_aekl3d": (1, 1, 8, 8, 8)}


def seg_onehot(shape, seed=0):
    """Deterministic one-hot segmentation map [N, label_nc, *spatial]."""
    import torch
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, shape[1], (shape[0], *shape[2:]), generator=g)
    return torch.nn.functional.one_hot(idx, shape[1]).movedim(-1, 1).float()


def head_channels_tuple(kw):
    n = len(kw["num_channels"])
    nhc = kw.get("num_head_channels", 8)
    return tuple(nhc) if isinstance(nhc, (tuple, list)) else (nhc,) * n


def unet_oracle_cfg(kw):
    return dict(num_head_channels=head_channels_tuple(kw), norm_num_groups=kw.get("norm_num_groups", 32),
                norm_eps=kw.get("norm_eps", 1e-6), with_conditioning=kw.get("with_conditioning", False))


def aekl_oracle_cfg(kw):
    return dict(norm_num_groups=kw.get("norm_num_groups", 32), norm_eps=kw.get("norm_eps", 1e-6),
                use_convtranspose=kw.get("use_convtranspose", False))


def vqvae_oracle_cfg(kw):
    return dict(downsample_parameters=kw["downsample_parameters"], upsample_parameters=kw["upsample_parameters"],
                commitment_cost=kw.get("commitment_cost", 0.25), output_act=kw.get("output_act"))


def randomize_zero_params(module, std=0.02, seed=1):
    """zero_module() leaves conv2 / proj_out / out convs all-zero; redraw them so parity tests are not vacuous
    (SURVEY.md §7 'reference quirks')."""
    import torch
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            if p.numel() > 0 and float(p.abs().max()) == 0.0:
                p.copy_(torch.randn(p.shape, generator=g) * std)
    return module


# brain-LDM bundle (model-zoo/.../configs/inference.json) at reduced widths: same topology and flags
BUNDLE_AEKL = dict(spatial_dims=3, in_channels=1, out_channels=1, latent_channels=3, num_channels=(8, 8, 16, 16),
                   num_res_blocks=2, norm_num_groups=4, norm_eps=1e-06, attention_levels=(False,) * 4,
                   with_encoder_nonlocal_attn=False, with_decoder_nonlocal_attn=False)
BUNDLE_UNET = dict(spatial_dims=3, in_channels=7, out_channels=3, num_channels=(8, 16, 16), num_res_blocks=2,
                   attention_levels=(False, True, True), norm_num_groups=8, norm_eps=1e-06, resblock_updown=True,
                   num_head_channels=(0, 16, 16), with_conditioning=True, transformer_num_layers=1,
                   cross_attention_dim=4, upcast_attention=True, use_flash_attention=False)
BUNDLE_SCHEDULER = dict(beta_start=0.0015, beta_end=0.0205, num_train_timesteps=1000, schedule="scaled_linear_beta",
                        clip_sample=False)
BUNDLE_STEPS = 5
BUNDLE_NOISE = (1, 3, 4, 8, 4)


# BASELINE.json configs[0] (C1): the reference's own CPU-runnable case — 2d_ddpm_tutorial.py:166-174 network,
# DDPMScheduler(1000) with set_timesteps(4), batch 2 of 1x64x64.  The 30 M weights are not committed: both sides
# regenerate them from this recipe (same state_dict keys and shapes on both sides).
C1_UNET = dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(128, 256, 256),
               attention_levels=(False, True, True), num_res_blocks=1, num_head_channels=256)
C1_SHAPE = (2, 1, 64, 64)
C1_STEPS = 4


def recipe_state_dict(module, seed=2024):
    """Deterministic, implementation-independent weights: every floating tensor of ``module.state_dict()`` (keys in
    sorted order) is drawn from one seeded CPU generator — matrices / filters ~ N(0, 1/fan_in), norm scales ~ 1 +
    0.1 N(0,1), biases ~ 0.1 N(0,1); integer buffers and attention masks keep their values.  Loads the result into
    ``module`` and returns it."""
    import math

    import torch
    g = torch.Generator().manual_seed(seed)
    sd = module.state_dict()
    out = {}
    for k in sorted(sd):
        t = sd[k]
        if not t.is_floating_point() or k.endswith("causal_mask"):
            out[k] = t.clone()
        elif t.dim() > 1:
            out[k] = torch.randn(t.shape, generator=g) / math.sqrt(t[0].numel())
        elif k.endswith("weight"):
            out[k] = 1.0 + 0.1 * torch.randn(t.shape, generator=g)
        else:
            out[k] = 0.1 * torch.randn(t.shape, generator=g)
    module.load_state_dict(out)
    return out


# BASELINE.json configs[1] (C2): 2d_ldm_tutorial.py:143-153 autoencoder + 303-311 latent UNet, DDIM-50 on a 3x64x64 latent
C2_AEKL = dict(spatial_dims=2, in_channels=1, out_channels=1, num_channels=(128, 128, 256), latent_channels=3,
               num_res_blocks=2, attention_levels=(False, False, False), with_encoder_nonlocal_attn=False,
               with_decoder_nonlocal_attn=False)
C2_UNET = dict(spatial_dims=2, in_channels=3, out_channels=3, num_res_blocks=2, num_channels=(128, 256, 512),
               attention_levels=(False, True, True), num_head_channels=(0, 256, 512))
C2_SCHEDULER = dict(num_train_timesteps=1000, schedule="linear_beta", beta_start=0.0015, beta_end=0.0195)
C2_LATENT = (1, 3, 64, 64)
C2_PROBES = (0, 1, 24, 49)             # DDIM step indices at which the reference trajectory is pinned teacher-forced


# BASELINE.json configs[2] (C3): 3d_ddpm_tutorial.py:159-167 network — the bench's headline model — at the tutorial's
# volume 32x40x32 (the oracle finishes a forward in seconds there): one forward + a DDIM-5 sample.  190 M weights from
# the recipe (seed 13), not committed.
C3_UNET = dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(256, 256, 512),
               attention_levels=(False, False, True), num_head_channels=(0, 0, 512), num_res_blocks=2)
C3_SCHEDULER = dict(num_train_timesteps=1000, schedule="scaled_linear_beta", beta_start=0.0005, beta_end=0.0195,
                    clip_sample=False)
C3_SHAPE = (1, 1, 32, 40, 32)
C3_STEPS = 5

# BASELINE.json configs[3] (C4): 3d_vqvae_tutorial.py:128-139 network at 1x64^3 (encode -> quantise -> decode)
C4_VQVAE = dict(spatial_dims=3, in_channels=1, out_channels=1, num_channels=(256, 256), num_res_channels=256,
                num_res_layers=2, downsample_parameters=((2, 4, 1, 1),) * 2,
                upsample_parameters=((2, 4, 1, 1, 0),) * 2, num_embeddings=256, embedding_dim=32)
C4_SHAPE = (1, 1, 64, 64, 64)

# BASELINE.json configs[4] (C5): 2d_controlnet.py:196-204 UNet widened to 3 channels with the CFG tutorial's
# cross-attention conditioning (classifier_free_guidance tutorial 193-203) + ControlNet (2d_controlnet.py:300-308),
# one classifier-free-guidance DDIM step at 3x256x256 (batch doubled to 2 inside the step; T = 16 384 at 128^2)
C5_COMMON = dict(spatial_dims=2, in_channels=3, num_res_blocks=1, num_channels=(128, 256, 256),
                 attention_levels=(False, True, True), num_head_channels=256, with_conditioning=True,
                 cross_attention_dim=1)
C5_UNET = dict(out_channels=3, **C5_COMMON)
C5_CONTROLNET = dict(conditioning_embedding_in_channels=1, conditioning_embedding_num_channels=(16,), **C5_COMMON)
C5_SHAPE = (1, 3, 256, 256)
C5_GUIDANCE = 7.0
C5_T_INDEX = 25           # DDIM-50 step index of the pinned step (t = 480)


def c5_mask():
    """Binary disc ((x-128)^2 + (y-128)^2 < 100^2), the synthetic control image of SURVEY.md section 8(d)."""
    import torch
    yy, xx = torch.meshgrid(torch.arange(256), torch.arange(256), indexing="ij")
    return (((xx - 128) ** 2 + (yy - 128) ** 2) < 100 ** 2).float()[None, None]
