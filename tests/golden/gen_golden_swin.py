"""Golden vectors for the Swin-T backbone + its FPN variant (SURVEY §8 a2): the reference's OWN
mmdet/models/backbones/swin_transformer.py::SwinTransformer (arguments of configs/dota/orientedrepoints_swin_tiny_demo.py:
9-25) and mmdet/models/necks/fpn.py::FPN(in_channels=[192,384,768], num_outs=5, GN) are imported from /root/reference and
run on the CPU in float64 (eval mode: DropPath is the identity).  Stubs: timm.models.layers (DropPath / to_2tuple /
trunc_normal_ - initialisers only, weights come from the state dict), mmcv_custom.load_checkpoint, registries.

    python tests/golden/gen_golden_swin.py     # needs /root/reference; writes tests/golden/swin_ref.npz
"""
import importlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import gen_golden_dense as gd                                                        # noqa: E402  (stubs for mmcv / mmdet plumbing)
from orientedreppoints_b200.swin import random_swin_state_dict                      # noqa: E402


def main():
    ResNet, FPN, Head = gd.install_stubs()
    timm = gd._pkg("timm")
    tm = gd._pkg("timm.models")
    layers = types.ModuleType("timm.models.layers")

    class DropPath(nn.Module):                                                       # identity in eval mode (timm/models/layers/drop.py)
        def __init__(self, drop_prob=None):
            super().__init__()

        def forward(self, x):
            return x
    layers.DropPath = DropPath
    layers.to_2tuple = lambda v: v if isinstance(v, tuple) else (v, v)
    layers.trunc_normal_ = lambda *a, **k: None
    sys.modules["timm.models.layers"] = layers
    timm.models, tm.layers = tm, layers
    mc = types.ModuleType("mmcv_custom")
    mc.load_checkpoint = lambda *a, **k: None
    sys.modules["mmcv_custom"] = mc
    Swin = importlib.import_module("mmdet.models.backbones.swin_transformer").SwinTransformer

    sd = random_swin_state_dict(0)
    backbone = Swin(embed_dim=96, depths=[2, 2, 6, 2], num_heads=[3, 6, 12, 24], window_size=7, mlp_ratio=4., qkv_bias=True,
                    qk_scale=None, drop_rate=0., attn_drop_rate=0., drop_path_rate=0.2, ape=False, patch_norm=True,
                    out_indices=(1, 2, 3), use_checkpoint=False)
    neck = FPN(in_channels=[192, 384, 768], out_channels=256, num_outs=5, norm_cfg=dict(type='GN', num_groups=32, requires_grad=True))
    m = nn.Module()
    m.backbone, m.neck = backbone, neck
    own = m.state_dict()
    given = {k: v for k, v in sd.items() if k.startswith(("backbone.", "neck."))}
    missing = [k for k in own if k not in given]
    unexpected = [k for k in given if k not in own]
    # buffers the reference derives itself (relative_position_index, attn_mask) may be absent from a checkpoint-style dict
    assert all(k.endswith(("relative_position_index", "attn_mask")) for k in missing), missing[:5]
    assert not unexpected, unexpected[:5]
    m.load_state_dict(given, strict=False)
    m = m.double().eval()
    out = {}
    for case, (h, w) in enumerate(((56, 84), (70, 100))):                            # the second needs window padding
        img = torch.randn(1, 3, h, w, generator=torch.Generator().manual_seed(20 + case), dtype=torch.float64)
        with torch.no_grad():
            c = m.backbone(img)
            f = m.neck(c)
        out["c%d_img" % case] = img.numpy()
        for i, t in enumerate(c):
            gd.store_sampled(out, "c%d_stage%d" % (case, i), t.numpy())
        for i, t in enumerate(f):
            gd.store_sampled(out, "c%d_fpn%d" % (case, i), t.numpy())
        print(case, [tuple(t.shape) for t in c], [tuple(t.shape) for t in f])
    np.savez_compressed(os.path.join(HERE, "swin_ref.npz"), **out)
    print("wrote swin_ref.npz")


if __name__ == "__main__":
    main()
