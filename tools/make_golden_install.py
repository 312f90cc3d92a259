"""Generate the fixtures of the drop-in tests: tests/golden/install_dit.pt, install_vae.pt and sampling_sigmas.json.

Runs the reference's own modules on CPU (WanModel of both trees, the two `WanVAE_` classes, hyvideo's AutoencoderKLCausal3D,
`get_sampling_sigmas` of fastvideo/sample/sample_5b.py) with the seeded weights and inputs of tests/test_host_logic*.py and
tests/test_sampler_host.py, and records what those tests compare with: the reference outputs, the state-dict layout of each
module and the attributes the install hooks read from it. The tests then run without the reference tree. Reference outputs are
stored in float16 (5e-4 relative rounding, far inside the bf16 budgets the tests apply) to keep the fixtures small.
    python tools/make_golden_install.py --reference <root of the reference checkout>
"""
from __future__ import annotations

import argparse
import ast
import importlib.util
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import make_golden  # noqa: E402
import make_golden_vae  # noqa: E402
from oracle import hyvae, synth, wan21vae, wan21vae_enc, wan22vae, wan22vae_enc  # noqa: E402

DIT_ATTRS = ("model_type", "dim", "ffn_dim", "num_heads", "num_layers", "in_dim", "out_dim", "text_len", "freq_dim", "patch_size", "eps")
WAN_VAE_ATTRS = ("dim", "z_dim", "dim_mult", "num_res_blocks", "temperal_downsample", "temperal_upsample")
HY_CONFIG = ("block_out_channels", "layers_per_block", "norm_num_groups", "sample_size", "sample_tsize", "latent_channels",
             "out_channels")
SIGMA_CASES = ((4, 7.0), (50, 3.0), (50, 5.0), (1, 7.0), (30, 1.0))


def layout(sd) -> dict:
    return {k: list(v.shape) for k, v in sd.items()}


def plain(v):
    return list(v) if isinstance(v, (list, tuple)) else v


@torch.no_grad()
def dit_fixtures() -> dict:
    """tests/test_host_logic_dit.py::test_install_on_the_reference_wanmodel_is_a_drop_in (weights 2468, inputs 77) and the layout
    check of tests/test_host_logic.py::test_install_on_the_reference_wanmodel_repacks_identically (weights 4321)."""
    out = {}
    for tree, cfg_name in (("wan23", "CFG_5B_TINY"), ("wan", "CFG_14B_TINY")):
        cfg = getattr(synth, cfg_name)
        mod = make_golden.load_reference(tree)
        model = make_golden.build_reference_model(mod, cfg, synth.make_state_dict(cfg, 2468))
        rec = {"layout": layout(model.state_dict()), "attrs": {a: plain(getattr(model, a)) for a in DIT_ATTRS},
               "has_img_emb": hasattr(model, "img_emb")}
        frames, H, W, lfz = 10 + 2, 6, 10, 2
        inp = synth.make_inputs(cfg, 77, frames, H, W, ctx_len=20)
        if cfg["variant"] == "5b":
            rec["want"] = model([inp["x"]], torch.tensor([[0.0, 400.0]]), [inp["context"]], seq_len=10 ** 6, latent_frame_zero=lfz,
                                flag=True)[0].half()
        else:
            rec["want"] = model([inp["x"]], torch.tensor([300.0]), [inp["context"]], seq_len=frames * (H // 2) * (W // 2),
                                clip_fea=inp["clip_fea"], y=[inp["y"]], rand_num_img=0.2, latent_frame_zero=lfz)[0].half()
        out[cfg_name] = rec
        print(tree, cfg_name, tuple(rec["want"].shape), len(rec["layout"]), "parameters")
    return out


def _load(path: Path, name: str):
    spec = importlib.util.spec_from_file_location(name, str(path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _wan_vae(model, wrapper_scale, video, z) -> dict:
    return {"layout": layout(model.state_dict()), "attrs": {a: plain(getattr(model, a)) for a in WAN_VAE_ATTRS},
            "want_mu": model.encode(video.unsqueeze(0), wrapper_scale).float().squeeze(0).half(),
            "want_x": model.decode(z.unsqueeze(0), wrapper_scale).float().clamp_(-1, 1).squeeze(0).half()}


@torch.no_grad()
def vae_fixtures(ref: Path) -> dict:
    """The three tests of tests/test_host_logic_vae_install.py, same seeds and inputs."""
    out = {}
    r22 = _load(ref / "wan23" / "modules" / "vae2_2.py", "ref_vae2_2_install")
    sd = dict(wan22vae_enc.make_state_dict(11, dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2,
                                           temperal_downsample=(False, True, True)))
    sd.update(wan22vae.make_state_dict(12, dec_dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_upsample=(True, True, False)))
    model = r22.WanVAE_(dim=32, dec_dim=32, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2, attn_scales=[],
                        temperal_downsample=[False, True, True]).eval()
    model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(3)
    mean, std = 0.3 * torch.randn(16, generator=g), 0.5 + torch.rand(16, generator=g)
    video = torch.randn(3, 5, 32, 64, generator=g).clamp_(-1, 1)
    z = torch.randn(16, 2, 2, 4, generator=g)
    out["wan22"] = _wan_vae(model, [mean, 1.0 / std], video, z)

    r21 = _load(ref / "wan" / "modules" / "vae.py", "ref_vae_install")
    cfg = dict(dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2)
    sd = dict(wan21vae_enc.make_state_dict(21, temperal_downsample=(False, True, True), **cfg))
    sd.update(wan21vae.make_state_dict(22, temperal_upsample=(True, True, False), **cfg))
    model = r21.WanVAE_(dim=32, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2, attn_scales=[], temperal_downsample=[False, True, True]).eval()
    model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(4)
    mean, std = 0.3 * torch.randn(16, generator=g), 0.5 + torch.rand(16, generator=g)
    video = torch.randn(3, 5, 16, 32, generator=g).clamp_(-1, 1)
    z = torch.randn(16, 2, 2, 4, generator=g)
    out["wan21"] = _wan_vae(model, [mean, 1.0 / std], video, z)

    make_golden_vae.REF = ref
    ak = make_golden_vae.load_reference_vae()
    cfg = make_golden_vae.TINY
    vae = ak.AutoencoderKLCausal3D(in_channels=3, out_channels=3, down_block_types=("DownEncoderBlockCausal3D",) * 4,
                                   up_block_types=("UpDecoderBlockCausal3D",) * 4, block_out_channels=cfg["block_out_channels"],
                                   layers_per_block=2, act_fn="silu", latent_channels=16, norm_num_groups=32, sample_size=64,
                                   sample_tsize=16, time_compression_ratio=4, spatial_compression_ratio=8, mid_block_add_attention=True)
    vae.load_state_dict(hyvae.make_state_dict(99, **cfg), strict=False)
    vae.eval()
    rec = {"layout": {k: s for k, s in layout(vae.state_dict()).items() if not k.startswith(("encoder.", "quant_conv."))},
           "config": {k: plain(getattr(vae.config, k)) for k in HY_CONFIG}}
    vae.enable_tiling()
    rec["tiling_on"] = (vae.use_spatial_tiling, vae.use_temporal_tiling)
    want = vae.decode(torch.randn(1, 16, 6, 10, 12, generator=torch.Generator().manual_seed(5)), return_dict=False)[0]
    # reduced like tests/golden/hyvae_tiny.pt: a stride-4 sample of the pixels plus full row / column sums (every pixel contributes)
    rec.update(shape=tuple(want.shape), sample=want[..., ::4, ::4].half(), rowsum=want.sum(-1).half(), colsum=want.sum(-2).half())
    vae.disable_tiling()
    rec["tiling_off"] = (vae.use_spatial_tiling, vae.use_temporal_tiling)
    rec["small_shape"] = tuple(vae.decode(torch.randn(1, 16, 2, 4, 6, generator=torch.Generator().manual_seed(6)), return_dict=False)[0].shape)
    out["hyvae"] = rec
    for k, v in out.items():
        print("vae", k, len(v["layout"]), "parameters")
    return out


def sampling_sigmas(ref: Path) -> list:
    """`get_sampling_sigmas` extracted from sample_5b.py (the script itself cannot be imported) at the tested (steps, shift)."""
    import numpy as np
    src = ref / "fastvideo" / "sample" / "sample_5b.py"
    tree = ast.parse(src.read_text())
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "get_sampling_sigmas")
    ns = {"np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), str(src), "exec"), ns)
    return [{"steps": s, "shift": sh, "sigmas": [float(x) for x in ns["get_sampling_sigmas"](s, sh)]} for s, sh in SIGMA_CASES]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, type=Path, help="root of the reference checkout (holds wan/, wan23/, hyvideo/)")
    args = ap.parse_args()
    torch.set_num_threads(8)
    make_golden.REF = args.reference
    gold = ROOT / "tests" / "golden"
    torch.save(dit_fixtures(), gold / "install_dit.pt")
    torch.save(vae_fixtures(args.reference), gold / "install_vae.pt")
    (gold / "sampling_sigmas.json").write_text(json.dumps(sampling_sigmas(args.reference), indent=1) + "\n")
    for name in ("install_dit.pt", "install_vae.pt", "sampling_sigmas.json"):
        print(name, (gold / name).stat().st_size, "bytes")


if __name__ == "__main__":
    main()
