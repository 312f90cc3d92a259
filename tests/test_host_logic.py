"""CPU tests of the host side: the C-ABI library exports, the FramePack plan, RoPE tables, error behaviour,
and the rule that nothing under yume_b200/ touches oracle/."""
import re
from pathlib import Path

import pytest
import torch

import yume_b200
from oracle import synth
from oracle.wan_dit import WanOracle, grid_freqs, rope_tables
from yume_b200 import _lib, ops
from yume_b200.dit import WanDiT, framepack_plan

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_header_symbol():
    header = (ROOT / "include" / "yume_b200.h").read_text()
    declared = set(re.findall(r"^\s*(?:int|long long)\s+(yb_\w+)\s*\(", header, flags=re.M))
    assert declared, "no declarations parsed"
    lib = yume_b200.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/yume_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), "ctypes signature table and header disagree"
    assert lib.yb_abi_version() == _lib.ABI_VERSION == 4


def test_ops_have_no_cpu_path():
    a = torch.zeros(128, 64, dtype=torch.bfloat16)
    with pytest.raises(yume_b200.YumeB200Error):
        ops.gemm(a, a, None, torch.zeros(128, 128, dtype=torch.bfloat16), ops.YB_EPI_BF16)
    with pytest.raises(yume_b200.YumeB200Error):
        ops.ln_modulate(torch.zeros(4, 64), torch.zeros(4, 64, dtype=torch.bfloat16), None, None)


def test_product_path_never_imports_oracle():
    for f in (ROOT / "yume_b200").rglob("*.py"):
        src = f.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f"{f} imports oracle/"
    for f in (ROOT / "yume_b200" / "csrc").glob("*"):
        if f.suffix in (".cu", ".cuh", ".h"):
            assert "oracle" not in f.read_text()


def _oracle_segments(variant, hist, branch_hist):
    m = WanOracle.__new__(WanOracle)
    m.variant = variant
    out = []
    for sl, name, padm, pre in m._segments(hist, branch_hist):
        start, stop, _ = sl.indices(hist)
        out.append((start, stop, name, pre))
    return out


@pytest.mark.parametrize("variant,lfz", [("5b", 8), ("14b", 9), ("14b", 8)])
def test_framepack_plan_matches_oracle_for_every_history_length(variant, lfz):
    lo = 1
    for hist in range(lo, 1367):
        branch = hist if variant == "5b" else hist + lfz - 9
        if branch > 1366:
            break
        try:
            want = _oracle_segments(variant, hist, branch)
        except IndexError:
            continue
        got = [(s.frames.start, s.frames.stop, s.name, s.pre_2x_f) for s in framepack_plan(hist, branch)]
        if any(a >= b or a < 0 for a, b, *_ in want):
            continue  # the reference itself indexes out of range / produces empty segments here
        assert got == want, (hist, got, want)


def test_framepack_plan_rejects_too_long_history():
    with pytest.raises(UnboundLocalError):
        framepack_plan(1400, 1400)


def _token_count(variant, frames, H, W, lfz):
    hist = frames - lfz
    plan = framepack_plan(hist, frames - (lfz if variant == "5b" else 9))
    n = 0
    for s in plan:
        f = s.frames.stop - s.frames.start
        n += f * -(-H // s.patch) * -(-W // s.patch)
    return n + lfz * (H // 2) * (W // 2)


def test_real_geometry_token_counts():
    # SURVEY.md §8: 5B FramePack chunk 13 latent frames @44x80 -> 9460; 14B @68x120 -> 21930 (lfz 8) / 23460 (lfz 9)
    assert _token_count("5b", 13, 44, 80, 8) == 9460
    assert _token_count("14b", 13, 68, 120, 8) == 21930
    assert _token_count("14b", 13, 68, 120, 9) == 23460
    assert 21 * 22 * 40 == 18480


@pytest.fixture(scope="module")
def tiny_engine_cpu():
    cfg = synth.CFG_5B_TINY
    sd = synth.make_state_dict(cfg, 1234)
    kw = synth.oracle_kwargs(cfg)
    kw.pop("variant")
    return WanDiT(sd, "5b", device="cpu", **kw)


def test_rope_table_matches_reference_tables(tiny_engine_cpu):
    eng = tiny_engine_cpu
    tabs = rope_tables(128)
    segs = [(1, 3, 5, 0), (2, 2, 3, 1), (4, 3, 5, 3)]
    want = torch.cat([grid_freqs(tabs, f, h, w, f0) for f, h, w, f0 in segs], dim=0).squeeze(1)  # complex128 [L, 64]
    got = eng._rope_table(segs)
    assert got.shape == (want.shape[0], 64, 2)
    assert torch.allclose(got[..., 0].double(), want.real, atol=1e-6)
    assert torch.allclose(got[..., 1].double(), want.imag, atol=1e-6)


def test_repack_layouts(tiny_engine_cpu):
    eng, C = tiny_engine_cpu, 256
    assert eng.blocks[0]["w_qkv"].shape == (3 * C, C) and eng.blocks[0]["w_qkv"].dtype == torch.bfloat16
    assert eng.block_mod.shape == (2, 6 * C)
    w, b = eng.embed["patch_embedding_2x_f"]
    assert w.shape == (64, 48 * 16) and b.shape == (64,)          # N padded 48 -> 64 for the GEMM tile
    assert eng.embed["patch_embedding_16x"][0].shape == (C, 48 * 32 * 32)


def test_mirror_state_dict_keys_match_reference_names():
    from yume_b200.model import WanModel14B, WanModel5B
    for cls, cfg in ((WanModel5B, synth.CFG_5B_TINY), (WanModel14B, synth.CFG_14B_TINY)):
        kw = dict(model_type="ti2v" if cfg["variant"] == "5b" else "i2v", text_len=cfg["text_len"], in_dim=cfg["in_dim"],
                  dim=cfg["dim"], ffn_dim=cfg["ffn_dim"], freq_dim=cfg["freq_dim"], text_dim=cfg["text_dim"],
                  out_dim=cfg["out_dim"], num_heads=cfg["num_heads"], num_layers=cfg["num_layers"])
        if cfg["variant"] == "14b":
            kw["clip_dim"] = cfg["clip_dim"]
        m = cls(**kw)
        have = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        want = synth.param_shapes(cfg)
        assert have == {k: tuple(v) for k, v in want.items()}


def test_wan22_vae_repack_folds_are_exact():
    """Host-side weight folding of the Wan2.2 VAE engine (no GPU): conv2 absorbs z*std+mean, proj absorbs the v bias."""
    import torch
    from oracle import wan22vae
    from yume_b200.vae22 import Wan22VaeDecoder, decoder_param_shapes
    cfg = dict(dec_dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_upsample=(True, True, False))
    assert decoder_param_shapes(**cfg) == wan22vae.param_shapes(**cfg)
    assert decoder_param_shapes() == wan22vae.param_shapes()
    sd = wan22vae.make_state_dict(3, **cfg)
    g = torch.Generator().manual_seed(0)
    mean, std = torch.randn(16, generator=g), 0.5 + torch.rand(16, generator=g)
    eng = Wan22VaeDecoder(sd, mean=mean, std=std, device="cpu", **cfg)
    z = torch.randn(7, 16, generator=g)
    w2, b2 = eng.lin["conv2"]
    want = (z * std + mean) @ sd["conv2.weight"].reshape(16, 16).T + sd["conv2.bias"]
    got = z @ w2.float()[:16, :16].T + b2[:16]
    assert float((got - want).norm() / want.norm()) < 1e-2          # bf16 weights
    assert bool((w2.float()[16:] == 0).all()) and bool((w2.float()[:, 16:] == 0).all())
    # time_conv split into two frame groups; Conv2d becomes (1,3,3) taps; every conv K is taps * Cp (Cp % 64 == 0)
    p = "decoder.upsamples.0.upsamples.3"
    assert eng.conv[p + ".time_conv.0"][2] == (3, 1, 1) and eng.conv[p + ".resample.1"][2] == (1, 3, 3)
    wt = sd[p + ".time_conv.weight"]
    C = wt.shape[1]
    w0 = eng.conv[p + ".time_conv.1"][0].float().view(C, 3, -1)[:, :, :C]
    assert torch.equal(w0, wt[C:, :, :, 0, 0].permute(0, 2, 1).bfloat16().float())
    for name, (w, b, taps) in eng.conv.items():
        assert w.shape[1] % (64 * taps[0] * taps[1] * taps[2]) == 0 and w.shape[0] % 32 == 0 and b.shape[0] == w.shape[0], name
    # v bias folded through proj
    a = "decoder.middle.1"
    Cq = eng.dims[0]
    Wo = sd[a + ".proj.weight"].reshape(Cq, Cq)
    assert torch.allclose(eng.att["bo"], sd[a + ".proj.bias"] + Wo @ sd[a + ".to_qkv.bias"][2 * Cq:], atol=1e-6)


def test_wan21_vae_plan_and_shapes_match_oracle():
    from oracle import wan21vae
    from yume_b200.vae21 import decoder_param_shapes, upsample_plan
    for dim in (96, 32):
        assert decoder_param_shapes(dim) == wan21vae.param_shapes(dim)
        assert upsample_plan(dim) == wan21vae.layer_plan(dim)
    kinds = [k for _, k, _, _ in upsample_plan()]
    assert kinds.count("upsample3d") == 2 and kinds.count("upsample2d") == 1 and kinds.count("res") == 12


class _FakeVaeModel:
    def __init__(self, sd, **attrs):
        self._sd = sd
        self.__dict__.update(attrs)

    def state_dict(self):
        return self._sd


def test_install_wan_vae_hooks_rebind_decode_with_reference_contract():
    """install_wan22_vae / install_wan21_vae read the wrapper's own attributes (vae2_2.py:748-792,909-1040;
    wan/modules/vae.py:484-500,618-645) and keep decode's list-in / list-out contract. No GPU: packing only."""
    import torch
    from oracle import wan21vae, wan22vae
    from yume_b200.vae21 import install_wan21_vae
    from yume_b200.vae22 import install_wan22_vae

    cfg22 = dict(dec_dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_upsample=(True, True, False))
    sd = wan22vae.make_state_dict(5, **cfg22)
    sd["encoder.conv1.weight"] = torch.zeros(4, 4, 3, 3, 3)          # encoder-side keys are ignored by the decode engine

    class W22:
        pass

    w = W22()
    w.model = _FakeVaeModel(sd, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2, temperal_upsample=[True, True, False])
    mean, std = torch.randn(16), 0.5 + torch.rand(16)
    w.scale = [mean, 1.0 / std]
    install_wan22_vae(w, device="cpu")
    eng = w._yb_decoder
    assert eng.dims == [128, 128, 128, 64, 32] and eng.z_dim == 16
    assert w.decode("not a list") is None                            # Wan2_2_VAE.decode logs a TypeError and returns None
    assert w.decode([]) == []
    w2, _ = eng.lin["conv2"]
    assert torch.allclose(w2.float()[:16, :16], (sd["conv2.weight"].reshape(16, 16) * std[None, :]).bfloat16().float())

    cfg21 = dict(dim=32, z_dim=16, dim_mult=(1, 2, 4, 4), num_res_blocks=2, temperal_upsample=(True, True, False))
    sd21 = wan21vae.make_state_dict(6, **cfg21)

    class W21:
        pass

    v = W21()
    v.model = _FakeVaeModel(sd21, dim=32, z_dim=16, dim_mult=[1, 2, 4, 4], num_res_blocks=2,
                            temperal_upsample=[True, True, False])
    v.mean, v.std = torch.randn(16), 0.5 + torch.rand(16)
    install_wan21_vae(v, device="cpu")
    assert v.decode([]) == [] and len(v._yb_decoder.plan) == 15
    with pytest.raises(Exception):
        v._yb_decoder.decode(torch.zeros(3, 1, 4, 4))               # wrong latent channel count is an error, not a guess


def test_wan_vae_param_shapes_match_reference_module_trees(golden_dir):
    """decoder_param_shapes() of both Wan VAE engines == the reference's own module trees at the real sizes
    (fixture: tools/make_golden_vae_shapes.py, built from vae2_2.py / vae.py on the meta device)."""
    import json
    from yume_b200 import vae21, vae22
    ref = json.loads((golden_dir / "wan_vae_shapes.json").read_text())
    assert {k: list(v) for k, v in vae22.decoder_param_shapes().items()} == ref["wan22"]
    assert {k: list(v) for k, v in vae21.decoder_param_shapes().items()} == ref["wan21"]


def test_attention_tail_split_plan():
    """Scheduler of the attention launch (host arithmetic exported as yb_attention_plan): the Ulysses per-rank shapes of
    the 720p step and the invariants the kernel relies on."""
    import ctypes as C
    from yume_b200 import _lib
    lib = _lib.load()

    def plan(Lq, Lk, heads, sms=148, flags=0):
        out = (C.c_int * 4)()
        assert lib.yb_attention_plan(Lq, Lk, heads, sms, flags, out) == 0
        return tuple(out)

    L = 18480
    assert plan(L, L, 3) == (148, 71, 2, 74)              # 8 GPUs: 219 units = 1.48 waves -> 71 tail units in two KV halves
    for heads in (24, 12, 6):                             # 1 / 2 / 4 GPUs: last wave more than half full, no split
        full, tail, ns, per = plan(L, L, heads)
        assert (tail, ns) == (0, 1) and full == heads * 73 and per == 145
    assert plan(L, L, 3, flags=2)[1] == 0                 # YB_ATT_ACCUMULATE launches never split
    assert plan(L, L, 3, flags=1 << 4)[1] == 0            # split policy 1 = never
    assert plan(300, 512, 2, flags=2 << 4) == (0, 4, 2, 2)    # forced: every unit, 4 key tiles -> 2 + 2
    assert plan(300, 256, 2, flags=2 << 4)[1] == 0            # too few key tiles to split
    assert lib.yb_attention_plan(0, 1, 1, 148, 0, (C.c_int * 4)()) != 0
    import itertools
    for Lq, Lk, heads, sms, force in itertools.product((1, 255, 257, 5000, 18480, 40000), (1, 129, 2049, 18480, 33000),
                                                       (1, 3, 5, 24), (1, 132, 148), (0, 2, 3, 4)):
        full, tail, ns, per = plan(Lq, Lk, heads, sms, flags=force << 4)
        units, nkv = ((Lq + 255) // 256) * heads, (Lk + 127) // 128
        assert full + tail == units and 1 <= ns <= 4 and (tail == 0) == (ns == 1)
        if ns > 1:
            assert per % 2 == 0 and (ns - 1) * per < nkv <= ns * per      # even segments, none empty, all keys covered
            if force == 0:
                assert full % sms == 0 and tail * ns <= sms               # the split tail fits in one wave


def test_conv_tile_plan():
    """Tile chooser of the implicit-GEMM conv (host arithmetic exported as yb_conv3d_plan) on the shapes of the three VAEs."""
    import ctypes as C
    from yume_b200 import _lib
    lib = _lib.load()

    def plan(T, H, W, cout, kw=3, fuse=0):
        out = (C.c_int * 4)()
        assert lib.yb_conv3d_plan(T, H, W, cout, kw, fuse, out) == 0
        return tuple(out)

    assert plan(21, 44, 80, 1024) == (16, 4, 2, 0)        # Wan2.2 level 0: a 128-wide row tile would waste 38 %
    assert plan(81, 176, 320, 512) == (64, 2, 1, 0)       # 256-wide N tile: fused only when the row tile is ~free
    assert plan(81, 352, 640, 256) == (128, 1, 1, 1)      # W multiple of 128: kw-fused halo mode
    assert plan(81, 544, 960, 96) == (128, 1, 1, 1)       # Wan2.1 96-channel level: fused (6 % ragged edge accepted)
    assert plan(81, 544, 960, 96, fuse=1)[3] == 0
    assert plan(40, 88, 160, 1024, kw=1)[3] == 0          # time_conv (3,1,1) has no kw taps to fuse
    assert plan(3, 8, 8, 64, fuse=2) == (128, 1, 1, 1)    # forced (tests): correct at any width, just wasteful
    assert plan(17, 256, 256, 128) == (128, 1, 1, 1)      # hyvideo last level
    for T, H, W, co in ((1, 1, 1, 32), (5, 3, 7, 64), (9, 4, 4, 32), (2, 130, 9, 64), (17, 32, 32, 512), (81, 720, 1280, 128)):
        tw, th, tt, fused = plan(T, H, W, co)
        assert tw * th * tt == 128 and tw <= max(128, 1)
        tiles = -(-W // tw) * -(-H // th) * -(-T // tt)
        assert tiles * 128 >= T * H * W
    assert lib.yb_conv3d_plan(1, 1, 1, 32, 2, 0, (C.c_int * 4)()) != 0


@pytest.mark.parametrize("tree,cfg_name", [("wan23", "CFG_5B_TINY"), ("wan", "CFG_14B_TINY")])
def test_install_on_the_reference_wanmodel_repacks_identically(golden_dir, tree, cfg_name):
    """Drop-in boundary (SURVEY.md §8b): `install()` on a live `WanModel` — a module with the parameter layout and attributes
    recorded from the REFERENCE's own class (tests/helpers/reference_modules.py) — must re-bind `forward` and build, from the
    module's own parameters (`WanDiT.from_module`), exactly the packed tensors the state-dict path builds."""
    from helpers import reference_modules
    from yume_b200 import model as ybm
    cfg = getattr(synth, cfg_name)
    sd = synth.make_state_dict(cfg, 4321)
    rec = torch.load(golden_dir / "install_dit.pt", weights_only=False)[cfg_name]
    ref_model = reference_modules.wanmodel(cfg, sd, rec)
    ref_forward = ref_model.forward
    ybm.install(ref_model, device="cpu")                               # repack only: no kernel runs at install time
    assert ref_model.forward is not ref_forward and ref_model.forward.__func__ in (ybm.forward_5b, ybm.forward_14b)
    eng = ref_model._yb_engine
    kw = synth.oracle_kwargs(cfg)
    want = WanDiT(sd, kw.pop("variant"), device="cpu", **kw)
    assert (eng.variant, eng.dim, eng.heads, eng.layers, eng.in_dim, eng.out_dim) == \
        (want.variant, want.dim, want.heads, want.layers, want.in_dim, want.out_dim)

    def same(a, b, path):
        if isinstance(a, torch.Tensor):
            assert a.dtype == b.dtype and torch.equal(a, b), path
        elif isinstance(a, dict):
            assert a.keys() == b.keys(), path
            for k in a:
                same(a[k], b[k], f"{path}.{k}")
        elif isinstance(a, (list, tuple)):
            assert len(a) == len(b), path
            for i, (x, y) in enumerate(zip(a, b)):
                same(x, y, f"{path}[{i}]")
    for name in ("embed", "text0", "text2", "time0", "time2", "tproj", "head_w", "head_b", "head_mod", "blocks", "block_mod",
                 "cw_kv_all", "cb_kv_all") + (("img", "cw_kv_img_all", "cb_kv_img_all") if cfg["variant"] == "14b" else ()):
        same(getattr(eng, name), getattr(want, name), name)
    # the re-bound forward keeps the reference's error behaviour without touching the GPU
    if cfg["variant"] == "14b":
        with pytest.raises(RuntimeError):
            ref_model([torch.zeros(16, 3, 8, 8)], torch.tensor([1.0]), [torch.zeros(4, 64)], 48, clip_fea=torch.zeros(1, 257, 96),
                      y=[torch.zeros(20, 3, 8, 8)], rand_num_img=None)
    else:
        with pytest.raises(NotImplementedError):
            ref_model([torch.zeros(48, 3, 8, 8)], torch.tensor([1.0]), [torch.zeros(4, 64)], 48, enable_mask=True)


def test_integration_doc_snippet_is_current():
    """INTEGRATION.md §3 shows the struct layouts a foreign caller must copy: the block is generated from the live binding
    and this test fails when either side changes without the other (round-1 ADVICE: a stale snippet over-read the struct)."""
    import sys
    sys.path.insert(0, str(ROOT / "tools"))
    import gen_integration_snippet as gen
    doc = (ROOT / "INTEGRATION.md").read_text()
    block = doc[doc.index(gen.BEGIN) + len(gen.BEGIN):doc.index(gen.END)].strip()
    assert block == gen.snippet().strip(), "run: python tools/gen_integration_snippet.py --write"


def test_ctypes_structs_match_the_c_header(tmp_path):
    """Compile include/yume_b200.h with gcc and compare sizeof / offsetof of both argument structs with the ctypes mirrors."""
    import ctypes as C
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = {"yb_gemm_args": _lib.GemmArgs, "yb_conv3d_args": _lib.Conv3dArgs}
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT / "include" / "yume_b200.h"}"', "int main(void) {"]
    for cname, cls in fields.items():
        prog.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            prog.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    prog += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in fields.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


def test_gemm_plan_kernel_choice():
    """Host-side kernel / tile choice of yb_gemm_bf16 (yb_gemm_plan): the SM-pair kernel with 256-wide tiles for the token GEMMs,
    the 1-CTA kernel for the small context / embedding projections."""
    import ctypes as C
    lib = yume_b200.load()
    out = (C.c_int * 4)()

    def plan(M, N):
        assert lib.yb_gemm_plan(M, N, 148, out) == 0
        return tuple(out)
    assert plan(18480, 3072) == (1, 256, 73, 12)
    assert plan(18480, 14336) == (1, 256, 73, 56)
    assert plan(2310, 9216) == (1, 256, 10, 36)
    assert plan(1024, 128) == (1, 128, 4, 1)
    assert plan(512, 3072) == (0, 256, 4, 12)            # context rows: 1-CTA kernel
    assert plan(257, 96) == (0, 128, 3, 1)
    assert lib.yb_gemm_plan(0, 128, 148, out) != 0


def test_gemm_tail_split_k_plan():
    """The split-K chooser of the SM-pair gate+residual GEMM (host arithmetic, no GPU): splits the per-rank shapes of 4- / 8-GPU
    Ulysses whose last wave is mostly idle, leaves full last waves and short-K launches alone, and every segment owns K blocks."""
    import ctypes as C
    lib = yume_b200.load()
    out = (C.c_int * 3)()

    def plan(tiles, num_kb, clusters=74, force=0):
        assert lib.yb_gemm_splitk_plan(tiles, num_kb, clusters, force, out) == 0
        return tuple(out)

    assert plan(120, 224)[1] == 1                 # 8 GPUs, FFN-down: 46 tail tiles need two sub-waves; measured gain 1 %: left alone
    assert plan(120, 224, force=3) == (74, 3, 75)
    assert plan(120, 48)[1] == 1                  # 8 GPUs, o-projection: the combine launch costs more than the idle tail
    full, ns, per = plan(228, 224)                # 4 GPUs, FFN-down: 6 tail tiles spread over the 74 pairs
    assert full == 222 and ns >= 6 and 6 * ns <= 74 and (ns - 1) * per < 224 <= ns * per
    assert plan(876, 224)[1] == 1 and plan(444, 224)[1] == 1     # 1 / 2 GPUs: last wave (nearly) full
    assert plan(74, 224) == (74, 1, 224) and plan(50, 224)[1] == 1
    assert plan(100, 224, force=2) == (74, 2, 112) and plan(100, 224, force=1)[1] == 1
    assert plan(5, 8, force=2) == (0, 2, 4) and plan(5, 3, force=2)[1] == 1
    for tiles in range(1, 400, 7):
        for num_kb in (8, 48, 80, 224):
            full, ns, per = plan(tiles, num_kb)
            assert 0 <= full <= tiles and 1 <= ns <= 12
            if ns > 1:
                assert full % 74 == 0 and (ns - 1) * per < num_kb <= ns * per and per >= 8


def test_graft_entry_build_runs():
    """The driver's CPU-side build check: __graft_entry__.build() compiles (no-op when the library is current), loads the
    library and checks the ABI version against the binding."""
    import importlib
    import sys
    sys.path.insert(0, str(ROOT))
    entry = importlib.import_module("__graft_entry__")
    entry.build()
