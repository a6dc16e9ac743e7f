"""SURVEY.md §8f rank 4 — the brain-LDM bundle edge (generativemodels_b200/bundle): the bundle's Sampler against the
fixture written by the reference's own scripts/sampler.py, the NIfTI writer against the standard's byte layout, the
inference.json resolver, and the packed-weight cache file.  CPU tests drive the real modules through the test-only
stand-in for the C-ABI (tests/cpu_backend.py); the ``gpu`` tests run the same checks on the CUDA path."""
import gzip
import json
import struct
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import torch_oracle as O
from tests import cpu_backend
from tests.golden import configs as G

GOLD = Path(__file__).resolve().parent / "golden"


def rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-12)).item()


def _bundle_models(device):
    from generativemodels_b200.networks.nets import AutoencoderKL, DiffusionModelUNet
    from generativemodels_b200.networks.schedulers import DDIMScheduler
    fx = torch.load(GOLD / "g_bundle_brain_ldm.pt", weights_only=False)
    ae = AutoencoderKL(**fx["aekl_kwargs"]).eval()
    unet = DiffusionModelUNet(**fx["unet_kwargs"]).eval()
    ae.load_state_dict(fx["aekl_state"])
    unet.load_state_dict(fx["unet_state"])
    sched = DDIMScheduler(**G.BUNDLE_SCHEDULER)
    sched.set_timesteps(num_inference_steps=G.BUNDLE_STEPS)
    return fx, ae.to(device), unet.to(device), sched


def _oracle_sample(fx):
    sched = O.DDIMOracle(**G.BUNDLE_SCHEDULER)
    sched.set_timesteps(G.BUNDLE_STEPS)
    ucfg, acfg = G.unet_oracle_cfg(fx["unet_kwargs"]), G.aekl_oracle_cfg(fx["aekl_kwargs"])
    return O.bundle_sampling_fn(
        lambda x, t, c: O.unet_forward(fx["unet_state"], ucfg, x, t, context=c),
        lambda z: O.autoencoderkl_decode(fx["aekl_state"], acfg, z), sched, fx["noise"], fx["conditioning"])


# ------------------------------------------------------------------------------------------------------------------
# oracle pinned to the reference's own bundle script
# ------------------------------------------------------------------------------------------------------------------
def test_oracle_bundle_sampler_matches_reference_fixture():
    fx = torch.load(GOLD / "g_bundle_brain_ldm.pt", weights_only=False)
    got = _oracle_sample(fx)
    assert got.shape == fx["sample"].shape
    assert rel(got, fx["sample"]) < 1e-5, rel(got, fx["sample"])


# ------------------------------------------------------------------------------------------------------------------
# host logic on the CPU stand-in
# ------------------------------------------------------------------------------------------------------------------
def test_bundle_sampler_golden_cpu(monkeypatch):
    cpu_backend.install(monkeypatch)
    from generativemodels_b200.bundle import Sampler
    fx, ae, unet, sched = _bundle_models("cpu")
    got = Sampler().sampling_fn(fx["noise"], ae, unet, sched, fx["conditioning"])
    assert got.shape == fx["sample"].shape and rel(got, fx["sample"]) < 5e-2, rel(got, fx["sample"])


def _parse_nifti(raw: bytes):
    assert struct.unpack_from("<i", raw, 0)[0] == 348 and raw[344:348] == b"n+1\0" and raw[348:352] == b"\0" * 4
    dim = struct.unpack_from("<8h", raw, 40)
    datatype, bitpix = struct.unpack_from("<hh", raw, 70)
    pixdim = struct.unpack_from("<8f", raw, 76)
    vox_offset = struct.unpack_from("<f", raw, 108)[0]
    slope, inter = struct.unpack_from("<ff", raw, 112)
    qcode, scode = struct.unpack_from("<hh", raw, 252)
    quat = struct.unpack_from("<6f", raw, 256)
    srow = np.array(struct.unpack_from("<12f", raw, 280)).reshape(3, 4)
    data = np.frombuffer(raw, np.uint8, offset=int(vox_offset)).reshape(dim[1:4], order="F")
    return dict(dim=dim, datatype=datatype, bitpix=bitpix, pixdim=pixdim, slope=slope, inter=inter, qcode=qcode,
                scode=scode, quat=quat, srow=srow, data=data)


def _check_saved(path, sample, saver):
    raw = gzip.open(path, "rb").read()
    f = _parse_nifti(raw)
    want = O.bundle_nifti_quantise(sample.cpu().numpy())
    assert f["dim"][0] == 3 and tuple(f["dim"][1:4]) == want.shape and f["datatype"] == 2 and f["bitpix"] == 8
    assert len(raw) == 352 + want.size
    assert np.array_equal(f["data"], want)                      # voxel [x, y, z] round-trips bit-exactly
    assert np.allclose(f["srow"], saver.affine[:3], atol=1e-5) and f["scode"] == 2 and f["qcode"] == 0
    assert f["pixdim"][0] == -1.0 and f["pixdim"][1:4] == (1.0, 1.0, 1.0)      # left-handed affine: qfac = -1
    assert np.allclose(f["quat"][:3], (0.0, 1.0, 0.0)) and np.allclose(f["quat"][3:], saver.affine[:3, 3], atol=1e-5)
    assert np.isnan(f["slope"]) and np.isnan(f["inter"])


def test_nifti_saver_cpu(tmp_path):
    from generativemodels_b200.bundle import NiftiSaver
    g = torch.Generator().manual_seed(3)
    sample = torch.randn(1, 1, 24, 30, 28, generator=g)
    saver = NiftiSaver(str(tmp_path))
    saver.save(sample, "vol")
    _check_saved(tmp_path / "vol.nii.gz", sample, saver)


def test_nifti_quaternion_is_the_affine_rotation():
    from generativemodels_b200.bundle.saver import _quaternion
    rng = np.random.default_rng(0)
    for _ in range(20):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        if q[0] < 0:
            q = -q
        a, b, c, d = q
        R = np.array([[a*a+b*b-c*c-d*d, 2*(b*c-a*d), 2*(b*d+a*c)],
                      [2*(b*c+a*d), a*a+c*c-b*b-d*d, 2*(c*d-a*b)],
                      [2*(b*d-a*c), 2*(c*d+a*b), a*a+d*d-b*b-c*c]])
        zooms = rng.uniform(0.5, 2.0, size=3)
        flip = rng.integers(0, 2) * 2 - 1
        A = np.eye(4)
        A[:3, :3] = R * zooms * np.array([1, 1, flip])
        qfac, qb, qc, qd, z = _quaternion(A)
        assert qfac == flip and np.allclose(z, zooms) and np.allclose((qb, qc, qd), (b, c, d), atol=1e-9)


_SMALL_CONFIG = {
    "imports": ["$import torch", "$from pathlib import Path"],
    "bundle_root": ".",
    "output_dir": "$@bundle_root + '/output'",
    "create_output_dir": "$Path(@output_dir).mkdir(exist_ok=True)",
    "age": 0.1,
    "conditioning": "$torch.tensor([[0.0, @age, 0.2, 0.4]]).unsqueeze(1)",
    "autoencoder_def": {"_target_": "generative.networks.nets.AutoencoderKL", **{
        k: (list(v) if isinstance(v, tuple) else v) for k, v in G.BUNDLE_AEKL.items()}},
    "load_autoencoder": "$@autoencoder_def.load_state_dict(@states['aekl_state'])",
    "autoencoder": "$@autoencoder_def.eval()",
    "diffusion_def": {"_target_": "generative.networks.nets.DiffusionModelUNet", **{
        k: (list(v) if isinstance(v, tuple) else v) for k, v in G.BUNDLE_UNET.items()}},
    "load_diffusion": "$@diffusion_def.load_state_dict(@states['unet_state'])",
    "diffusion": "$@diffusion_def.eval()",
    "scheduler": {"_target_": "generative.networks.schedulers.DDIMScheduler",
                  "_requires_": ["@load_diffusion", "@load_autoencoder"], **G.BUNDLE_SCHEDULER},
    "set_timesteps": "$@scheduler.set_timesteps(num_inference_steps=%d)" % G.BUNDLE_STEPS,
    "sampler": {"_target_": "scripts.sampler.Sampler", "_requires_": "@set_timesteps"},
    "sample": "$@sampler.sampling_fn(@states['noise'], @autoencoder, @diffusion, @scheduler, @conditioning)",
    "saver": {"_target_": "scripts.saver.NiftiSaver", "_requires_": "@create_output_dir", "output_dir": "@output_dir"},
    "save_nii": "$@saver.save(@sample, 'out')",
}


def test_bundle_config_runs_reference_syntax_cpu(monkeypatch, tmp_path):
    """Same item graph as the bundle's inference.json (targets in the reference's namespace, ``_requires_`` ordering,
    ``@`` references inside ``$`` expressions), resolved onto the B200 classes."""
    cpu_backend.install(monkeypatch)
    from generativemodels_b200.bundle import BundleConfig, NiftiSaver, Sampler
    from generativemodels_b200.networks.nets import AutoencoderKL
    fx = torch.load(GOLD / "g_bundle_brain_ldm.pt", weights_only=False)
    cfg = BundleConfig(json.loads(json.dumps(_SMALL_CONFIG)), {"bundle_root": str(tmp_path), "states": "$None"})
    cfg._resolved["states"] = fx                               # tensors cannot come through JSON
    cfg.run("save_nii")
    assert isinstance(cfg.get("autoencoder"), AutoencoderKL) and isinstance(cfg.get("sampler"), Sampler)
    assert isinstance(cfg.get("saver"), NiftiSaver) and cfg.get("sample") is cfg.get("sample")
    assert rel(cfg.get("sample"), fx["sample"]) < 5e-2
    _check_saved(tmp_path / "output" / "out.nii.gz", cfg.get("sample"), cfg.get("saver"))
    # overrides and error behaviour
    assert BundleConfig(dict(_SMALL_CONFIG), {"age": 0.7}).get("conditioning")[0, 0, 1].item() == pytest.approx(0.7)
    with pytest.raises(KeyError):
        cfg.get("nope")
    with pytest.raises(ValueError, match="circular"):
        BundleConfig({"a": "@b", "b": "$@a + 1"}).get("a")
    assert BundleConfig({"x": {"_target_": "collections.OrderedDict", "_disabled_": True}}).get("x") is None
    assert BundleConfig({"l": [1, {"k": 5}], "v": "@l#1#k", "w": "$@l::1::k + 1"}).run("v", "w") == [5, 6]


def test_reference_inference_json_parses_when_present():
    """The unmodified bundle config (configs/inference.json of the model zoo's
    brain_image_synthesis_latent_diffusion_model, stored as tests/golden/brain_ldm_inference.json) resolves its network
    definitions on this package."""
    path = GOLD / "brain_ldm_inference.json"
    from generativemodels_b200.bundle import BundleConfig, Sampler
    from generativemodels_b200.networks.nets import AutoencoderKL, DiffusionModelUNet
    from generativemodels_b200.networks.schedulers import DDIMScheduler
    cfg = BundleConfig(str(path), {"load_autoencoder": "$None", "load_diffusion": "$None", "device": "$'cpu'",
                                   "diffusion_def#num_channels": [32, 64, 64],
                                   "diffusion_def#num_head_channels": [0, 64, 64]})
    ae = cfg.get("autoencoder")
    assert isinstance(ae, AutoencoderKL) and tuple(cfg.get("noise").shape) == (1, 3, 20, 28, 20)
    assert isinstance(cfg.get("scheduler"), DDIMScheduler) and isinstance(cfg.get("sampler"), Sampler)
    assert len(cfg.get("scheduler").timesteps) == 50 and tuple(cfg.get("conditioning").shape) == (1, 1, 4)
    assert isinstance(cfg.get("diffusion"), DiffusionModelUNet) and cfg.get("diffusion").in_channels == 7


def test_bundle_cli_cpu(tmp_path, capsys):
    """``python -m generativemodels_b200.bundle run <ids> --config_file f --key value`` (monai.bundle's call shape)."""
    from generativemodels_b200.bundle.__main__ import main
    cfg = tmp_path / "c.json"
    cfg.write_text(json.dumps({"imports": ["$from pathlib import Path"], "root": ".", "age": 0.1, "name": "a",
                               "touch": "$Path(@root, @name + str(@age)).write_text('x')"}))
    assert main(["run", "touch", "--config_file", str(cfg), "--root", str(tmp_path), "--age", "0.7"]) == 0
    assert (tmp_path / "a0.7").read_text() == "x"
    assert main(["run", "touch", "--config_file", str(cfg), "--root", str(tmp_path), "--name", "b"]) == 0
    assert (tmp_path / "b0.1").exists()
    assert main([]) == 2 and main(["run", "--config_file", str(cfg)]) == 2 and main(["run", "touch"]) == 2
    assert main(["run", "touch", "--config_file"]) == 2
    capsys.readouterr()


def test_packed_cache_roundtrip_cpu(monkeypatch, tmp_path):
    cpu_backend.install(monkeypatch)
    from generativemodels_b200 import ops
    from generativemodels_b200.bundle import fingerprint, load_packed, save_packed
    from generativemodels_b200.networks.nets import DiffusionModelUNet
    fx, _, unet, _ = _bundle_models("cpu")
    x = torch.cat([fx["noise"], torch.zeros(1, 4, *fx["noise"].shape[2:])], 1)
    t = torch.tensor([500])
    want = unet(x, t, context=fx["conditioning"])
    n = save_packed(unet, str(tmp_path / "unet.packed.pt"))
    assert n > 20
    fresh = DiffusionModelUNet(**fx["unet_kwargs"]).eval()
    fresh.load_state_dict(fx["unet_state"])
    assert fingerprint(fresh) == fingerprint(unet)
    assert load_packed(fresh, str(tmp_path / "unet.packed.pt"))
    built = []
    for cls in ("PackedConv", "PackedLinear", "PackedUpsampleConv", "PackedConvTranspose"):
        orig = getattr(ops, cls).__init__
        monkeypatch.setattr(getattr(ops, cls), "__init__",
                            lambda self, *a, _o=orig, _c=cls, **k: (built.append(_c), _o(self, *a, **k))[1])
    got = fresh(x, t, context=fx["conditioning"])
    assert torch.equal(got, want) and built == []              # nothing was repacked
    # different weights: refused, and the lazily packed result reflects the NEW weights
    other = DiffusionModelUNet(**fx["unet_kwargs"]).eval()
    other.load_state_dict(fx["unet_state"])
    with torch.no_grad():
        next(other.parameters()).mul_(1.5)
    assert not load_packed(other, str(tmp_path / "unet.packed.pt"))
    assert not torch.equal(other(x, t, context=fx["conditioning"]), want) and built


# ------------------------------------------------------------------------------------------------------------------
# CUDA path
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_bundle_sampler_golden_gpu(graph):
    from generativemodels_b200.bundle import Sampler
    fx, ae, unet, sched = _bundle_models("cuda")
    got = Sampler(use_cuda_graph=graph).sampling_fn(fx["noise"].cuda(), ae, unet, sched, fx["conditioning"].cuda())
    torch.cuda.synchronize()
    # bf16 activations through 5 x UNet + a 4-level decoder vs the reference's fp32 CPU run
    assert got.shape == fx["sample"].shape and rel(got.cpu(), fx["sample"]) < 5e-2, rel(got.cpu(), fx["sample"])


@pytest.mark.gpu
def test_nifti_saver_gpu_bytes_equal_numpy_restatement(tmp_path):
    from generativemodels_b200.bundle import NiftiSaver
    g = torch.Generator().manual_seed(3)
    sample = torch.randn(1, 1, 40, 44, 48, generator=g)
    saver = NiftiSaver(str(tmp_path))
    saver.save(sample.cuda(), "vol")
    _check_saved(tmp_path / "vol.nii.gz", sample, saver)      # device arithmetic == numpy arithmetic, bit for bit


@pytest.mark.gpu
def test_packed_cache_roundtrip_gpu(tmp_path):
    from generativemodels_b200.bundle import load_packed, save_packed
    from generativemodels_b200.networks.nets import AutoencoderKL
    fx, ae, _, _ = _bundle_models("cuda")
    z = fx["noise"].cuda()
    want = ae.decode_stage_2_outputs(z)
    assert save_packed(ae, str(tmp_path / "ae.packed.pt")) > 10
    fresh = AutoencoderKL(**fx["aekl_kwargs"]).eval()
    fresh.load_state_dict(fx["aekl_state"])
    fresh = fresh.cuda()
    assert load_packed(fresh, str(tmp_path / "ae.packed.pt"))
    assert torch.equal(fresh.decode_stage_2_outputs(z), want)
