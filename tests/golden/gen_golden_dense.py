"""Golden vectors for the dense graph (SURVEY §8 a1, a3, a4, a5): the reference's OWN modules

    mmdet/models/backbones/resnet.py        ResNet(depth=50 | 101, style='pytorch')
    mmdet/models/necks/fpn.py               FPN(start_level=1, add_extra_convs=True, num_outs=5, GN)
    mmdet/ops/conv_module.py, norm.py, conv.py, activation.py
    mmdet/models/anchor_heads/orientedreppoints_head.py   OrientedRepPointsHead.__init__/_init_layers/forward(_single)

are imported FROM /root/reference and executed on the CPU in float64, built with the arguments of
configs/dota/orientedrepoints_r50_demo.py:4-44 and loaded (strict=True: same key names) with the state dict
`orientedreppoints_b200.weights.random_state_dict` produces.  The mmdet package itself cannot be imported (mmcv 0.6.2 is
absent), so its plumbing is stubbed: `mmcv.cnn` initialisers (weights are overwritten by the state dict), the registries,
`auto_fp16`, loss builders; the ONE compute stub is `DeformConv` (CUDA-only extension in the reference), replaced by
oracle/torch_reference.py::deform_conv_ref (itself an im2col restatement of deform_conv_cuda_kernel.cu).

    python tests/golden/gen_golden_dense.py     # needs /root/reference; writes tests/golden/dense_r50.npz
"""
import importlib
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import torch_reference as tr                                             # noqa: E402
from orientedreppoints_b200.weights import random_state_dict                        # noqa: E402


def _pkg(name, path=None):
    m = types.ModuleType(name)
    m.__path__ = [path] if path else []
    sys.modules[name] = m
    return m


def install_stubs():
    ident = lambda *a, **k: None                                                     # noqa: E731
    mmcv = _pkg("mmcv")
    cnn = types.ModuleType("mmcv.cnn")
    for n in ("constant_init", "kaiming_init", "xavier_init", "normal_init"):
        setattr(cnn, n, ident)
    runner = types.ModuleType("mmcv.runner")
    runner.load_checkpoint = ident
    sys.modules["mmcv.cnn"], sys.modules["mmcv.runner"] = cnn, runner
    mmcv.cnn, mmcv.runner = cnn, runner

    mmdet = _pkg("mmdet", os.path.join(REF, "mmdet"))

    class Registry:
        def register_module(self, cls=None):                                         # used both as @R.register_module and @R.register_module()
            return cls if cls is not None else (lambda c: c)
    utils = types.ModuleType("mmdet.utils")
    utils.get_root_logger = lambda *a, **k: None
    utils.Registry = Registry
    sys.modules["mmdet.utils"] = utils
    mmdet.utils = utils

    # mmdet.ops: the real conv_module / conv / norm / activation / conv_ws files, DeformConv replaced
    ops = _pkg("mmdet.ops", os.path.join(REF, "mmdet", "ops"))

    class DeformConv(nn.Module):
        """stand-in for mmdet/ops/dcn/deform_conv.py:DeformConv (CUDA extension): same parameters (weight, no bias), forward
        through the oracle's im2col restatement"""

        def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                     deformable_groups=1, bias=False):
            super().__init__()
            assert not bias and groups == 1 and deformable_groups == 1
            self.stride, self.padding, self.dilation = stride, padding, dilation
            self.weight = nn.Parameter(torch.zeros(out_channels, in_channels, kernel_size, kernel_size))

        def forward(self, x, offset):
            return tr.deform_conv_ref(x, offset, self.weight, self.stride, self.padding, self.dilation)

    dcn = types.ModuleType("mmdet.ops.dcn")
    dcn.DeformConv = DeformConv
    dcn.DeformConvPack = dcn.ModulatedDeformConvPack = type("Unused", (nn.Module,), {})
    sys.modules["mmdet.ops.dcn"] = dcn
    mar = types.ModuleType("mmdet.ops.minarearect")
    mar.minaerarect = None
    cd = types.ModuleType("mmdet.ops.chamfer_distance")
    cd.ChamferDistance2D = type("ChamferDistance2D", (), {})
    sys.modules["mmdet.ops.minarearect"], sys.modules["mmdet.ops.chamfer_distance"] = mar, cd
    conv_module = importlib.import_module("mmdet.ops.conv_module")                  # REAL reference files from here on
    conv = importlib.import_module("mmdet.ops.conv")
    norm = importlib.import_module("mmdet.ops.norm")
    ops.ConvModule, ops.build_conv_layer, ops.build_norm_layer = conv_module.ConvModule, conv.build_conv_layer, norm.build_norm_layer
    ops.DeformConv, ops.ContextBlock, ops.GeneralizedAttention = DeformConv, None, None

    core = _pkg("mmdet.core")
    pg = importlib.util.spec_from_file_location("mmdet.core.anchor.point_generator",
                                                os.path.join(REF, "mmdet/core/anchor/point_generator.py"))
    pgm = importlib.util.module_from_spec(pg)
    pg.loader.exec_module(pgm)                                                        # REAL PointGenerator

    def multi_apply(func, *args, **kwargs):                                          # mmdet/core/utils/misc.py:32-36
        from functools import partial
        pfunc = partial(func, **kwargs) if kwargs else func
        return tuple(map(list, zip(*map(pfunc, *args))))
    core.auto_fp16 = lambda *a, **k: (lambda f: f)
    core.force_fp32 = lambda *a, **k: (lambda f: f)
    core.PointGenerator, core.multi_apply, core.multiclass_rnms, core.levels_to_images = pgm.PointGenerator, multi_apply, None, None
    bbox = types.ModuleType("mmdet.core.bbox")
    bbox.init_pointset_target = bbox.refine_pointset_target = None
    sys.modules["mmdet.core.bbox"] = bbox
    core.bbox = bbox

    models = _pkg("mmdet.models", os.path.join(REF, "mmdet", "models"))
    reg = types.ModuleType("mmdet.models.registry")
    reg.BACKBONES = reg.NECKS = reg.HEADS = Registry()
    builder = types.ModuleType("mmdet.models.builder")
    builder.build_loss = lambda cfg: None
    sys.modules["mmdet.models.registry"], sys.modules["mmdet.models.builder"] = reg, builder
    models.registry, models.builder = reg, builder
    for sub in ("backbones", "necks", "anchor_heads"):
        _pkg("mmdet.models." + sub, os.path.join(REF, "mmdet", "models", sub))
    return (importlib.import_module("mmdet.models.backbones.resnet").ResNet,
            importlib.import_module("mmdet.models.necks.fpn").FPN,
            importlib.import_module("mmdet.models.anchor_heads.orientedreppoints_head").OrientedRepPointsHead)


def build_reference_model(ResNet, FPN, Head, depth):
    gn = dict(type='GN', num_groups=32, requires_grad=True)
    backbone = ResNet(depth=depth, num_stages=4, out_indices=(0, 1, 2, 3), frozen_stages=1,
                      norm_cfg=dict(type='BN', requires_grad=True), style='pytorch')
    neck = FPN(in_channels=[256, 512, 1024, 2048], out_channels=256, start_level=1, add_extra_convs=True, num_outs=5, norm_cfg=gn)
    head = Head(num_classes=16, in_channels=256, feat_channels=256, point_feat_channels=256, stacked_convs=3, num_points=9,
                gradient_mul=0.3, point_strides=[8, 16, 32, 64, 128], point_base_scale=2, norm_cfg=gn,
                loss_cls=dict(type='FocalLoss', use_sigmoid=True, gamma=2.0, alpha=0.25, loss_weight=1.0),
                loss_rbox_init=dict(type='GIoULoss', loss_weight=0.375), loss_rbox_refine=dict(type='GIoULoss', loss_weight=1.0),
                loss_spatial_init=dict(type='SpatialBorderLoss', loss_weight=0.05),
                loss_spatial_refine=dict(type='SpatialBorderLoss', loss_weight=0.1), top_ratio=0.4)
    m = nn.Module()
    m.backbone, m.neck, m.bbox_head = backbone, neck, head
    return m


SAMPLE = 4096


def store_sampled(out, key, a):
    """store the output `a` as at most SAMPLE of its elements at fixed, seeded flat positions (key_idx) together with its
    shape (key_shape): the test still runs the whole graph, and every golden file stays under 1 MB"""
    if a.size <= SAMPLE:
        idx = np.arange(a.size)
    else:
        idx = np.sort(np.random.RandomState(0).choice(a.size, SAMPLE, replace=False))
    out[key] = a.reshape(-1)[idx]
    out[key + "_idx"] = idx.astype(np.int32)
    out[key + "_shape"] = np.array(a.shape, dtype=np.int64)


def main():
    ResNet, FPN, Head = install_stubs()
    out = {}
    for depth, (h, w), seed in ((50, (96, 128), 0), (101, (64, 96), 3)):
        sd = random_state_dict(depth, seed=seed, reference_init=False)
        model = build_reference_model(ResNet, FPN, Head, depth)
        missing = model.load_state_dict(sd, strict=True)                              # the reference's own key names
        assert not missing.missing_keys and not missing.unexpected_keys
        model = model.double().eval()
        img = torch.randn(1, 3, h, w, generator=torch.Generator().manual_seed(seed + 10), dtype=torch.float64)
        with torch.no_grad():
            feats = model.neck(model.backbone(img))
            cls, init, refine, _ = model.bbox_head(feats)
        tag = "r%d" % depth
        out[tag + "_meta"] = np.array([depth, seed, h, w], dtype=np.int64)
        out[tag + "_img"] = img.numpy()
        for l in range(5):
            store_sampled(out, "%s_feat%d" % (tag, l), feats[l].numpy())
            store_sampled(out, "%s_cls%d" % (tag, l), cls[l].numpy())
            store_sampled(out, "%s_init%d" % (tag, l), init[l].numpy())
            store_sampled(out, "%s_refine%d" % (tag, l), refine[l].numpy())
        print(tag, [tuple(f.shape) for f in feats], float(feats[0].abs().max()), float(cls[0].abs().max()))
    np.savez_compressed(os.path.join(HERE, "dense_ref.npz"), **out)
    print("wrote dense_ref.npz")


if __name__ == "__main__":
    main()
