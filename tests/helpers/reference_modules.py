"""Stand-ins for the reference's own modules in the drop-in tests, checked against what tools/make_golden_install.py recorded from
those modules (tests/golden/install_*.pt): the same state-dict keys and shapes, and the same values of every attribute an install
hook reads. The hooks see nothing else of a module, so over a stand-in that passes these checks they take the path they take
on the reference's module."""
import types

import torch

DIT_ATTRS = ("model_type", "dim", "ffn_dim", "num_heads", "num_layers", "in_dim", "out_dim", "text_len", "freq_dim", "patch_size", "eps")


def plain(v):
    return list(v) if isinstance(v, (list, tuple)) else v


def check_layout(sd, rec) -> None:
    assert {k: list(v.shape) for k, v in sd.items()} == rec["layout"], "state-dict keys / shapes differ from the reference module"


def wanmodel(cfg: dict, sd: dict, rec: dict) -> torch.nn.Module:
    """yume_b200.model's WanModel5B / WanModel14B built like the reference's `WanModel(...)`, with `sd` loaded into real parameters."""
    from yume_b200.model import WanModel5B, WanModel14B
    kw = dict(text_len=cfg["text_len"], in_dim=cfg["in_dim"], dim=cfg["dim"], ffn_dim=cfg["ffn_dim"], freq_dim=cfg["freq_dim"],
              text_dim=cfg["text_dim"], out_dim=cfg["out_dim"], num_heads=cfg["num_heads"], num_layers=cfg["num_layers"], eps=1e-6)
    if cfg["variant"] == "5b":
        m = WanModel5B(model_type="ti2v", **kw)
    else:
        m = WanModel14B(model_type="i2v", clip_dim=cfg["clip_dim"], **kw)
    m.load_state_dict(sd, strict=True)
    check_layout(m.state_dict(), rec)
    assert {a: plain(getattr(m, a)) for a in DIT_ATTRS} == rec["attrs"] and hasattr(m, "img_emb") == rec["has_img_emb"]
    return m.eval()


def module(sd: dict, rec: dict, **attrs) -> types.SimpleNamespace:
    """A module-like object holding `sd` (its state dict) and `attrs`, after checking both against the recorded reference module."""
    check_layout(sd, rec)
    assert {k: plain(v) for k, v in attrs.items()} == rec.get("attrs", {}), "attributes differ from the reference module"
    return types.SimpleNamespace(state_dict=lambda: dict(sd), **attrs)
