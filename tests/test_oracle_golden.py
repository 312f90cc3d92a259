"""Pin the CPU oracle (oracle/wan_dit.py) against outputs of the reference's own WanModel code.

tests/golden/*.pt were produced by tools/make_golden.py, which imports /root/reference/wan{,23}/modules/model.py
in the authoring container. Same seeded weights/inputs (oracle/synth.py), same CPU fp32 regime -> the restatement
must agree to fp32 round-off."""
import pytest
import torch

from oracle import synth
from oracle.wan_dit import WanOracle

TOL = 2e-5  # fp32 accumulation-order noise only


@pytest.fixture(autouse=True)
def _golden_thread_count():
    """Run with the 8 intra-op threads tools/make_golden.py generated the goldens with. The thread count sets how CPU kernels split
    fp32 reductions, and the bf16 attention inputs turn that last-bit difference into ~3e-4 on the dim-1024 models at 16 or more
    threads; with the generator's count the oracle reproduces the reference's sums."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def _load(golden_dir, name):
    g = torch.load(golden_dir / name, weights_only=False)
    sd = synth.make_state_dict(g["cfg"], g["seed_w"])
    got = float(sum(v.abs().sum() for v in sd.values()))
    if abs(got - g["weight_abs_sum"]) > 1e-3 * g["weight_abs_sum"]:
        pytest.skip("torch CPU RNG stream differs from the one that generated the golden weights")
    return g, sd


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.fixture(scope="module")
def g5(golden_dir):
    return _load(golden_dir, "wan23_tiny.pt")


@pytest.fixture(scope="module")
def g14(golden_dir):
    return _load(golden_dir, "wan21_tiny.pt")


@pytest.mark.parametrize("case", ["5b_grid", "5b_grid_padded", "5b_pack_h3", "5b_pack_h1", "5b_pack_h10",
                                  "5b_pack_h30", "5b_pack_h100", "5b_pack_h400"])
def test_5b_forward_matches_reference(g5, case):
    g, sd = g5
    c = g["cases"][case]
    cfg = g["cfg"]
    inp = synth.make_inputs(cfg, c["seed"], c["frames"], c["H"], c["W"], c["ctx_len"])
    m = WanOracle(sd, **synth.oracle_kwargs(cfg))
    out = m.forward([inp["x"]], torch.tensor(c["t"]), [inp["context"]], seq_len=c["seq_len"],
                    latent_frame_zero=c["lfz"], flag=c["flag"])
    assert out.shape == c["out"].shape
    assert _rel(out, c["out"]) < TOL


def test_5b_block_matches_reference(g5):
    g, sd = g5
    cfg, b = g["cfg"], g["block"]
    gen = torch.Generator().manual_seed(b["seed"])
    L, C = b["L"], cfg["dim"]
    x = torch.randn(1, L, C, generator=gen)
    e = 0.5 * torch.randn(1, L, 6, C, generator=gen)
    ctx = torch.randn(1, cfg["text_len"], C, generator=gen)
    m = WanOracle(sd, **synth.oracle_kwargs(cfg))
    from oracle.wan_dit import grid_freqs
    y = m.block(0, x, e, grid_freqs(m.tables, *b["grid"]), ctx)
    assert _rel(y, b["out"]) < TOL


@pytest.mark.parametrize("case", ["14b_grid", "14b_pack_h4", "14b_pack_lfz8", "14b_pack_h12"])
def test_14b_forward_matches_reference(g14, case):
    g, sd = g14
    c = g["cases"][case]
    cfg = g["cfg"]
    inp = synth.make_inputs(cfg, c["seed"], c["frames"], c["H"], c["W"], c["ctx_len"])
    m = WanOracle(sd, **synth.oracle_kwargs(cfg))
    out = m.forward([inp["x"]], torch.tensor(c["t"]), [inp["context"]], seq_len=c["seq_len"], y=[inp["y"]],
                    clip_fea=inp["clip_fea"], latent_frame_zero=c["lfz"], rand_num_img=c["rand_num_img"])
    assert out.shape == c["out"].shape
    assert _rel(out, c["out"]) < TOL


def test_history_beyond_last_branch_raises(g5):
    g, sd = g5
    m = WanOracle(sd, **synth.oracle_kwargs(g["cfg"]))
    with pytest.raises(UnboundLocalError):
        m._segments(1400, 1400)


# 8-head models (dim 1024): the goldens the Ulysses parity runs at world 2 / 4 / 8 use (tools/sp_parity.py)
def _h8(golden_dir, name):
    g = torch.load(golden_dir / name, weights_only=False)
    return g, synth.make_state_dict(g["cfg"], g["seed_w"])


@pytest.mark.parametrize("case", ["5b_grid", "5b_grid_padded", "5b_pack_h10", "5b_pack_h30"])
def test_5b_h8_forward_matches_reference(golden_dir, case):
    g, sd = _h8(golden_dir, "wan23_h8.pt")
    c, cfg = g["cases"][case], g["cfg"]
    inp = synth.make_inputs(cfg, c["seed"], c["frames"], c["H"], c["W"], c["ctx_len"])
    out = WanOracle(sd, **synth.oracle_kwargs(cfg)).forward([inp["x"]], torch.tensor(c["t"]), [inp["context"]],
                                                            seq_len=c["seq_len"], latent_frame_zero=c["lfz"], flag=c["flag"])
    assert out.shape == c["out"].shape and _rel(out, c["out"]) < TOL


@pytest.mark.parametrize("case", ["14b_grid", "14b_grid_padded", "14b_pack_lfz8"])
def test_14b_h8_forward_matches_reference(golden_dir, case):
    """14b_grid_padded: seq_len > F*H*W — the 14B tree masks the padded rows as keys (k_lens = seq_lens,
    wan/modules/model.py:311-314, 916); the 5B tree does not (5b_grid_padded above)."""
    g, sd = _h8(golden_dir, "wan21_h8.pt")
    c, cfg = g["cases"][case], g["cfg"]
    inp = synth.make_inputs(cfg, c["seed"], c["frames"], c["H"], c["W"], c["ctx_len"])
    out = WanOracle(sd, **synth.oracle_kwargs(cfg)).forward([inp["x"]], torch.tensor(c["t"]), [inp["context"]],
                                                            seq_len=c["seq_len"], y=[inp["y"]], clip_fea=inp["clip_fea"],
                                                            latent_frame_zero=c["lfz"], rand_num_img=c["rand_num_img"])
    assert out.shape == c["out"].shape and _rel(out, c["out"]) < TOL
