"""Drop-in hooks of the Wan VAEs and the hyvideo VAE on CPU: `install_*` on a wrapper holding a module with the parameter layout and the
attributes of the REFERENCE's own class (`WanVAE_` of the 2.2 and 2.1 trees, `AutoencoderKLCausal3D`; tests/helpers/reference_modules.py),
held the way `Wan2_2_VAE` / `WanVAE` hold it (`.model`, `.scale` / `.mean`, `.std`; their constructors want a checkpoint file), then
`encode(list)` / `decode(list)` — list in / list out, outputs within the bf16 budget of what the reference's own chunked encode / decode
computed from the same seeded weights and inputs (tests/golden/install_vae.pt, tools/make_golden_install.py). The engines run over the
torch stand-in for the C ABI (tests/helpers/torch_ops.py)."""
import types

import pytest
import torch

from helpers import reference_modules, torch_ops
from oracle import wan21vae, wan21vae_enc, wan22vae, wan22vae_enc
from yume_b200 import vae21, vae22, vae_enc


@pytest.fixture()
def cpu_ops(monkeypatch):
    for mod in (vae22, vae21, vae_enc):
        monkeypatch.setattr(mod, "ops", torch_ops)


@pytest.fixture(scope="module")
def recorded(golden_dir):
    return torch.load(golden_dir / "install_vae.pt", weights_only=False)


def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm())


@torch.no_grad()
def test_wan22_wrapper_hooks_are_drop_ins(cpu_ops, recorded):
    rec = recorded["wan22"]
    cfg = dict(dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_downsample=(False, True, True))
    sd = dict(wan22vae_enc.make_state_dict(11, **cfg))
    sd.update(wan22vae.make_state_dict(12, dec_dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_upsample=(True, True, False)))
    model = reference_modules.module(sd, rec, dim=32, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2,
                                     temperal_downsample=[False, True, True], temperal_upsample=[True, True, False])
    g = torch.Generator().manual_seed(3)
    mean, std = 0.3 * torch.randn(16, generator=g), 0.5 + torch.rand(16, generator=g)
    wrapper = types.SimpleNamespace(model=model, scale=[mean, 1.0 / std], dtype=torch.float)
    video = torch.randn(3, 5, 32, 64, generator=g).clamp_(-1, 1)
    z = torch.randn(16, 2, 2, 4, generator=g)
    want_mu, want_x = rec["want_mu"], rec["want_x"]
    vae_enc.install_wan22_vae_encoder(wrapper, device="cpu")
    vae22.install_wan22_vae(wrapper, device="cpu")
    got_mu, got_x = wrapper.encode([video]), wrapper.decode([z])
    assert isinstance(got_mu, list) and isinstance(got_x, list) and len(got_mu) == len(got_x) == 1
    assert got_mu[0].shape == want_mu.shape and _rel(got_mu[0], want_mu) < 3e-2
    assert got_x[0].shape == want_x.shape and _rel(got_x[0], want_x) < 3e-2
    assert wrapper.encode(video) is None and wrapper.decode(z) is None          # the reference logs a TypeError and returns None


@torch.no_grad()
def test_wan21_wrapper_hooks_are_drop_ins(cpu_ops, recorded):
    rec = recorded["wan21"]
    cfg = dict(dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2)
    sd = dict(wan21vae_enc.make_state_dict(21, temperal_downsample=(False, True, True), **cfg))
    sd.update(wan21vae.make_state_dict(22, temperal_upsample=(True, True, False), **cfg))
    model = reference_modules.module(sd, rec, dim=32, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2,
                                     temperal_downsample=[False, True, True], temperal_upsample=[True, True, False])
    g = torch.Generator().manual_seed(4)
    mean, std = 0.3 * torch.randn(16, generator=g), 0.5 + torch.rand(16, generator=g)
    wrapper = types.SimpleNamespace(model=model, mean=mean, std=std, scale=[mean, 1.0 / std], dtype=torch.float)
    video = torch.randn(3, 5, 16, 32, generator=g).clamp_(-1, 1)
    z = torch.randn(16, 2, 2, 4, generator=g)
    want_mu, want_x = rec["want_mu"], rec["want_x"]
    vae_enc.install_wan21_vae_encoder(wrapper, device="cpu")
    vae21.install_wan21_vae(wrapper, device="cpu")
    got_mu, got_x = wrapper.encode([video]), wrapper.decode([z])
    assert got_mu[0].shape == want_mu.shape and _rel(got_mu[0], want_mu) < 3e-2
    assert got_x[0].shape == want_x.shape and _rel(got_x[0], want_x) < 3e-2


@torch.no_grad()
def test_hyvideo_install_vae_is_a_drop_in(monkeypatch, recorded):
    """`install_vae` on an `AutoencoderKLCausal3D` (the reference's config and decoder layout, its `enable_tiling()` /
    `disable_tiling()` switch values as recorded): the re-bound `decode(z, return_dict=...)` — same return convention, tiling
    honoured, output within the bf16 budget of the module's own tiled decode."""
    from oracle import hyvae
    from yume_b200 import vae as ybvae
    monkeypatch.setattr(ybvae, "ops", torch_ops)
    rec = recorded["hyvae"]
    cfg = dict(block_out_channels=(64, 64, 128, 128), layers_per_block=2, latent_channels=16, out_channels=3)
    sd = hyvae.make_state_dict(99, **cfg)
    ref = reference_modules.module(sd, rec)
    ref.config = types.SimpleNamespace(norm_num_groups=32, sample_size=64, sample_tsize=16, **cfg)
    assert {k: reference_modules.plain(getattr(ref.config, k)) for k in rec["config"]} == rec["config"]
    ref.use_spatial_tiling, ref.use_temporal_tiling = rec["tiling_on"]           # enable_tiling()
    z = torch.randn(1, 16, 6, 10, 12, generator=torch.Generator().manual_seed(5))
    ybvae.install_vae(ref, device="cpu")

    def check(dec):
        assert tuple(dec.shape) == rec["shape"]
        for key, got in (("sample", dec[..., ::4, ::4]), ("rowsum", dec.sum(-1)), ("colsum", dec.sum(-2))):
            assert _rel(got, rec[key]) < 3e-2, key
    got = ref.decode(z, return_dict=False)
    assert isinstance(got, tuple)
    check(got[0])
    check(ref.decode(z).sample)
    ref.use_spatial_tiling, ref.use_temporal_tiling = rec["tiling_off"]          # disable_tiling(): the hook follows the module's switches
    small = torch.randn(1, 16, 2, 4, 6, generator=torch.Generator().manual_seed(6))
    assert ref.decode(small, return_dict=False)[0].shape == rec["small_shape"] == (1, 3, 5, 32, 48)
