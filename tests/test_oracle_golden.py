"""CPU: the oracle (oracle/*.c) against the golden vectors minted from the reference itself
(tests/golden/gen_golden*.py).  Bit-exact: the oracle restates the reference's arithmetic operation for operation."""
import os

import numpy as np
import pytest


def test_unit_squares_one_seventh(po):
    # the only known answer the reference itself carries (DOTA_devkit/polyiou.cpp:130-136)
    p = np.array([0, 0, 1, 0, 1, 1, 0, 1], np.float64)
    q = p + 0.5
    assert po.iou_poly_f64(p, q)[0] == 0.14285714285714285
    assert abs(float(po.iou_rnms_f32(p, q)[0]) - 1.0 / 7.0) < 1e-6


def test_iou_pairs_bit_exact_vs_reference(po, golden):
    g = golden("iou_pairs.npz")
    o64 = po.iou_poly_f64(g["p"], g["q"])
    o32 = po.iou_rnms_f32(g["p"], g["q"])
    assert np.array_equal(o64, g["ref64"], equal_nan=True)          # polyiou.cpp, fp64
    assert np.array_equal(o32, g["ref32"], equal_nan=True)          # rnms_cpu.cpp rotate_iou, fp32
    assert (g["ref64"] > 1e-6).sum() > 2000                         # the fixture is not trivially disjoint


@pytest.mark.parametrize("name", ["nms_1k.npz", "nms_clustered.npz", "nms_1k_offset16000.npz"])
def test_nms_keep_sets_vs_reference(po, golden, name):
    g = golden(name)
    d = g["dets"]
    for thr, key in ((0.1, "keep64_thr01"), (0.3, "keep64_thr03")):
        assert np.array_equal(po.nms_poly_f64(d, thr), g[key])      # py_cpu_nms_poly + SWIG polyiou
    assert np.array_equal(po.nms_poly_f64(d, 0.1, fast=True), g["keep64fast_thr01"])
    for thr, key in ((0.1, "keep32_thr01"), (0.4, "keep32_thr04")):
        assert np.array_equal(po.nms_f32(d, np.float32(thr)), g[key])  # rnms_cpu.soft_rnms(method=0)


def test_fp32_reference_is_unstable_far_from_origin(golden):
    """SURVEY H1, documented deviation: the reference's fp32 path keeps 511 of the boxes its own fp64
    path keeps 660 of, once every coordinate is shifted by +16000 (what the class-offset trick does)."""
    near, far = golden("nms_1k.npz"), golden("nms_1k_offset16000.npz")
    assert len(near["keep32_thr01"]) == len(near["keep64_thr01"]) == 660
    assert len(far["keep64_thr01"]) == 660 and len(far["keep32_thr01"]) == 511


def test_clustered_iou_pairs_bit_exact_vs_reference(po, golden):
    # pairs drawn from object-like clusters; the reference's polyiou.cpp (fp64) and rotate_iou (fp32) outputs are stored
    g = golden("iou_clustered.npz")
    d = g["dets"]
    p, q = d[g["i"], :8], d[g["j"], :8]
    assert np.array_equal(po.iou_poly_f64(p, q), g["ref64"], equal_nan=True)
    assert np.array_equal(po.iou_rnms_f32(p, q), g["ref32"], equal_nan=True)
    assert (g["ref64"] > 1e-6).sum() >= 100                        # the fixture is not trivially disjoint


def test_guard_and_nan_conventions(po):
    z = np.zeros(8, np.float32)
    assert np.isnan(po.iou_rnms_f32(z, z)[0])                       # rnms: 0/0
    assert po.iou_polynms_f32_one(z, z) == 1.0                      # poly_nms guard: (0+1)/(0+1)


def test_poly_overlaps_oracle_matches_fp64_on_corners(po):
    rng = np.random.RandomState(0)
    b = np.stack([rng.uniform(0, 200, 64), rng.uniform(0, 200, 64), rng.uniform(8, 64, 64),
                  rng.uniform(4, 32, 64), rng.uniform(-1.5, 1.5, 64)], 1).astype(np.float32)
    o = po.poly_overlaps_f32(b[:32], b[32:])
    qa, qb = po.rotbox_to_quad_f32(b[:32]), po.rotbox_to_quad_f32(b[32:])
    ref = po.iou_poly_f64_matrix(qa, qb)
    assert np.abs(o - ref).max() < 5e-3   # the reference's own fp32 error at these coordinates


# --------------------------------------------------------------------------- minarearect oracle
def _area(b):
    b = b.reshape(-1, 4, 2).astype(np.float64)
    x, y = b[:, :, 0], b[:, :, 1]
    return 0.5 * np.abs((x * np.roll(y, -1, 1) - y * np.roll(x, -1, 1)).sum(1))


def test_minarearect_oracle_properties(po):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.RandomState(0)
    pts = rng.normal(0, 3, (3000, 9, 2)).astype(np.float32)
    box, hmap, hn = po.minarearect(pts.reshape(-1, 18))
    a = _area(box)
    ac = np.array([(lambda r: r[1][0] * r[1][1])(cv2.minAreaRect(p)) for p in pts])
    assert np.max(np.abs(a - ac) / ac) < 1e-5                      # same minimum area as OpenCV
    # every input point lies inside the rectangle
    b = box.reshape(-1, 4, 2).astype(np.float64)
    e = np.roll(b, -1, 1) - b
    for k in range(4):
        d = pts - b[:, k:k + 1, :]
        cr = e[:, k:k + 1, 0] * d[:, :, 1] - e[:, k:k + 1, 1] * d[:, :, 0]
        sg = np.sign(np.median(cr))
        assert (cr * sg > -1e-3).all()
    # hull map points at input points that are hull vertices
    assert ((hn >= 3) & (hn <= 9)).all()
    for i in range(50):
        idx = hmap[i, :hn[i]]
        assert (idx >= 0).all() and len(set(idx.tolist())) == hn[i]


def test_minarearect_oracle_analytic(po):
    # axis-aligned 2x1 rectangle + interior points: corners in the reference's order
    # (xmax,ymin),(xmin,ymin),(xmin,ymax),(xmax,ymax)  (minarearect_kernel.cu:380-450)
    p = np.array([[0, 0, 2, 0, 2, 1, 0, 1, 1, 0.5, 1, 0.2, 0.5, 0.5, 1.5, 0.5, 1, 0.8]], np.float32)
    box, hmap, hn = po.minarearect(p)
    assert hn[0] == 4 and list(hmap[0, :4]) == [0, 1, 2, 3]
    assert np.allclose(box[0], [2, 0, 0, 0, 0, 1, 2, 1], atol=1e-6)
    # all points identical -> a degenerate rectangle at that point
    box, _, hn = po.minarearect(np.full((1, 18), 3.0, np.float32))
    assert np.allclose(box, 3.0, atol=1e-5)


def _convex_cases(po, n, k, seed):
    rng = np.random.RandomState(seed)
    pts = (rng.rand(n, 9, 2) * 60 + rng.rand(n, 1, 2) * 100).astype(np.float32)
    quads = po.gen_rotated_boxes(k, seed=seed + 1, extent=160.0, wmin=10, wmax=80)[:, :8].astype(np.float32)
    return pts.reshape(n, 18), quads


def test_convex_iou_oracle_agrees_with_opencv(po):
    """the convex_iou restatement (mmdet/ops/iou/src/convex_iou_kernel.cu:139-312; CUDA-only in the reference, so
    unpinned by it) against an independent implementation: cv2.convexHull + cv2.intersectConvexConvex"""
    cv2 = pytest.importorskip("cv2")
    pts, quads = _convex_cases(po, 120, 25, 0)
    out = po.convex_iou(pts, quads)
    assert out.shape == (120, 25) and out.dtype == np.float32
    worst = 0.0
    for i in range(pts.shape[0]):
        hull = cv2.convexHull(pts[i].reshape(9, 2)).reshape(-1, 2)
        ha = cv2.contourArea(hull)
        ring = po.convex_hull9(pts[i])
        assert ring.shape[0] == hull.shape[0]                       # same hull vertices (general position)
        for j in range(quads.shape[0]):
            q = quads[j].reshape(4, 2)
            ia, _ = cv2.intersectConvexConvex(hull.astype(np.float32), q)
            iou = ia / (ha + cv2.contourArea(q) - ia)
            worst = max(worst, abs(iou - float(out[i, j])))
    assert worst < 1e-5, worst
    assert (out > 0.05).mean() > 0.05                               # the cases do overlap


def test_convex_iou_oracle_analytic(po):
    # 9 points on/in the unit square -> hull is the square; IoU with the shifted unit square = 1/7 (polyiou.cpp:130-136)
    sq = np.array([0, 0, 1, 0, 1, 1, 0, 1, .5, .5, .5, 0, 1, .5, .5, 1, 0, .5], dtype=np.float32)
    q = np.array([[.5, .5, 1.5, .5, 1.5, 1.5, .5, 1.5], [0, 0, 1, 0, 1, 1, 0, 1], [5, 5, 6, 5, 6, 6, 5, 6]], dtype=np.float32)
    out = po.convex_iou(sq[None], q)[0]
    assert abs(out[0] - 1.0 / 7.0) < 1e-7 and abs(out[1] - 1.0) < 1e-7 and out[2] == 0.0
    # orientation of the quadrilateral does not matter (intersectAreaO reverses clockwise rings, :128-129)
    assert po.convex_iou(sq[None], q[:1, [0, 1, 6, 7, 4, 5, 2, 3]])[0, 0] == out[0]


def test_result_merge_restatement_equals_reference_output(po):
    """SURVEY 8 n1: tile-level Task1 lines -> coordinates back to the image -> per-image poly NMS (thr 0.1) -> merged lines.
    tests/golden/result_merge.json was produced by the reference's OWN ResultMerge_multi_process.mergesingle
    (py_cpu_nms_poly_fast and py_cpu_nms_poly, over the SWIG polyiou compiled from its polyiou.cpp); the restatement
    (result_merge.parse_result_lines + the fp64 CPU oracle NMS + the reference's line format) reproduces every line."""
    import json
    from orientedreppoints_b200.dota import result_merge as rm
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "result_merge.json")))
    assert g["nms_thresh"] == rm.nms_thresh == 0.1
    names, ids, dets = rm.parse_result_lines(g["lines"])
    assert names == ["P0003", "P0007", "P0011"] or sorted(names) == ["P0003", "P0007", "P0011"]
    exp = []
    for k, name in enumerate(names):                              # dict order = first appearance (mergesingle :190-213)
        idx = np.nonzero(ids == k)[0]
        for fast in (True, False):
            keep = po.nms_poly_f64(dets[idx], g["nms_thresh"], fast=fast)
            if fast:
                keep_fast = keep
            else:
                assert np.array_equal(keep, keep_fast)
        for i in idx[keep_fast]:
            exp.append(name + ' ' + str(float(dets[i, 8])) + ' ' + ' '.join(map(str, [float(v) for v in dets[i, :8]])))
    assert exp == g["merged"]
    assert 1000 < len(exp) < len(g["lines"])


@pytest.mark.parametrize("case", [0, 1, 2, 3])
def test_postprocess_restatement_equals_reference_python(case):
    """SURVEY 8 a7 + a9: tests/golden/postprocess.npz holds what the reference's OWN get_bboxes_single
    (orientedreppoints_head.py:707-779) and multiclass_rnms (bbox_nms.py:93-182) return - extracted with ast and executed by
    tests/golden/gen_golden_postprocess.py with minaerarect / rnms replaced by their CPU oracles.  The restatement the GPU
    path is checked against (oracle/torch_reference.py::get_bboxes_single: class segments instead of the coordinate-offset
    trick, stable sorts) reproduces detections, labels and their order exactly."""
    import torch
    from oracle import torch_reference as tr
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "postprocess.npz"))
    seed, thr, pre, cap = g["c%d_cfg" % case]
    cls = [torch.from_numpy(g["c%d_cls%d" % (case, l)]) for l in range(5)]
    pts = [torch.from_numpy(g["c%d_pts%d" % (case, l)]) for l in range(5)]
    d, l = tr.get_bboxes_single(cls, pts, nms_pre=int(pre), score_thr=float(thr), iou_thr=0.4, max_per_img=int(cap))
    assert d.shape[0] > 0 and d.shape[1] == 27
    assert np.array_equal(d.numpy(), g["c%d_dets" % case]) and np.array_equal(l.numpy(), g["c%d_labels" % case])


def _assert_sampled_close(t, g, key):
    """float64 output `t` against the reference output stored as a fixed sample of its elements (key_idx: flat positions,
    key_shape: full shape; tests/golden/gen_golden_dense.py::store_sampled), to rounding noise"""
    ref = g[key]
    assert tuple(t.shape) == tuple(g[key + "_shape"]), key
    a = t.reshape(-1).numpy()[g[key + "_idx"]]
    assert np.abs(a - ref).max() < 1e-10 * max(1.0, np.abs(ref).max()), key


@pytest.mark.parametrize("depth", [50, 101])
def test_dense_graph_restatement_equals_reference_modules(depth):
    """SURVEY 8 a1/a3/a4/a5: tests/golden/dense_ref.npz holds the outputs of the reference's OWN ResNet, FPN and
    OrientedRepPointsHead modules (imported from /root/reference by tests/golden/gen_golden_dense.py with mmcv/registry
    plumbing stubbed and DeformConv replaced by the oracle's deform_conv_ref), loaded with strict=True from
    weights.random_state_dict (same key names) and run in float64.  The functional restatement the GPU engines are checked
    against (oracle/torch_reference.py::forward_dense) agrees to rounding noise on every FPN level and head output (outputs
    of more than 4096 elements are stored and compared at 4096 fixed positions)."""
    import torch
    from oracle import torch_reference as tr
    from orientedreppoints_b200.weights import STAGE_BLOCKS, random_state_dict
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "dense_ref.npz"))
    tag = "r%d" % depth
    d, seed, h, w = [int(v) for v in g[tag + "_meta"]]
    sd = {k: v.double() for k, v in random_state_dict(d, seed=seed, reference_init=False).items()}
    img = torch.from_numpy(g[tag + "_img"])
    with torch.no_grad():
        outs, feats = tr.forward_dense(sd, img, blocks=STAGE_BLOCKS[d])
    for l in range(5):
        _assert_sampled_close(feats[l], g, "%s_feat%d" % (tag, l))
        for k, n in enumerate(("cls", "init", "refine")):
            _assert_sampled_close(outs[l][k], g, "%s_%s%d" % (tag, n, l))


@pytest.mark.parametrize("case", [0, 1])
def test_swin_restatement_equals_reference_module(case):
    """SURVEY 8 a2: tests/golden/swin_ref.npz holds the outputs of the reference's OWN SwinTransformer
    (backbones/swin_transformer.py, arguments of configs/dota/orientedrepoints_swin_tiny_demo.py:9-25) and FPN
    (in_channels [192,384,768], num_outs 5, GN), imported from /root/reference by tests/golden/gen_golden_swin.py (timm /
    mmcv plumbing stubbed) and run in float64; case 1 exercises the window padding.  The functional restatement the GPU
    Swin path is checked against (oracle/torch_swin.py) agrees to rounding noise (outputs of more than 4096 elements are
    stored and compared at 4096 fixed positions)."""
    import torch
    from oracle import torch_swin as ts
    from orientedreppoints_b200.swin import random_swin_state_dict
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "swin_ref.npz"))
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in random_swin_state_dict(0).items()}
    img = torch.from_numpy(g["c%d_img" % case])
    with torch.no_grad():
        c = ts.swin_forward(sd, img)
        f = ts.swin_fpn(sd, c)
    assert len(c) == 3 and len(f) == 5
    for i, a in enumerate(c):
        _assert_sampled_close(a, g, "c%d_stage%d" % (case, i))
    for i, a in enumerate(f):
        _assert_sampled_close(a, g, "c%d_fpn%d" % (case, i))


def test_dcn_oracle_agrees_with_torchvision():
    """SURVEY 8 a6: the reference's DeformConv is a CUDA-only extension (mmdet/ops/dcn/src/deform_conv_cuda_kernel.cu), so
    the im2col restatement the GPU kernels are checked against cannot be pinned by the reference itself.  It is pinned
    against an independent implementation of the same operator (torchvision.ops.deform_conv2d, CPU): same offset layout
    (dy, dx per tap), same zero-outside bilinear rule, DCNv1 and DCNv2 (mask), strides / paddings / dilations."""
    tv = pytest.importorskip("torchvision.ops")
    import torch
    from oracle import torch_reference as tr
    g = torch.Generator().manual_seed(0)
    for (n, c, h, w, co, s, p, d) in [(2, 8, 11, 13, 6, 1, 1, 1), (1, 16, 9, 9, 4, 2, 1, 1), (1, 4, 10, 12, 5, 1, 2, 2),
                                      (1, 8, 7, 8, 8, 1, 0, 1)]:
        x = torch.randn(n, c, h, w, generator=g, dtype=torch.float64)
        wt = torch.randn(co, c, 3, 3, generator=g, dtype=torch.float64)
        ho, wo = (h + 2 * p - 2 * d - 1) // s + 1, (w + 2 * p - 2 * d - 1) // s + 1
        off = torch.randn(n, 18, ho, wo, generator=g, dtype=torch.float64) * 2.5     # many samples leave the image
        m = torch.rand(n, 9, ho, wo, generator=g, dtype=torch.float64)
        a = tr.deform_conv_ref(x, off, wt, s, p, d)
        b = tv.deform_conv2d(x, off, wt, None, stride=s, padding=p, dilation=d)
        assert a.shape == b.shape and float((a - b).abs().max()) < 1e-10
        a = tr.deform_conv_ref(x, off, wt, s, p, d, mask=m)
        b = tv.deform_conv2d(x, off, wt, None, stride=s, padding=p, dilation=d, mask=m)
        assert float((a - b).abs().max()) < 1e-10


def _quad_area(b):
    b = b.reshape(-1, 4, 2).astype(np.float64)
    x, y = b[..., 0], b[..., 1]
    return 0.5 * np.abs((x * np.roll(y, -1, 1) - y * np.roll(x, -1, 1)).sum(1))


def test_minarearect_oracle_vs_reference_device_code(po):
    """SURVEY 8 a8: tests/golden/device_ops_ref.npz holds what the reference's OWN __device__ code of
    minarearect_kernel.cu (Findminbox / Jarvis_and_index, compiled as host C++ by oracle/build_ref.py) returns.
    Hull index maps: identical.  Rectangles: identical or within 2e-6 (the reference calls cosf, the oracle and the CUDA
    kernel evaluate cos in double and round - DESIGN deviation 3), except near-ties of the min-area argmin (< 0.1 % of the
    sets) where the other, equally small rectangle is chosen: same area to 1e-6."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "device_ops_ref.npz"))
    boxes, maps, hull_n = po.minarearect(g["mar_pts"])
    assert np.array_equal(hull_n, g["mar_hull_n"])
    for i in range(len(hull_n)):
        assert np.array_equal(maps[i][:hull_n[i]], g["mar_map"][i][:hull_n[i]]), i
    d = np.abs(boxes - g["mar_boxes"]).max(1)
    scale = np.maximum(1.0, np.abs(g["mar_boxes"]).max(1))
    ties = np.nonzero(d > 2e-6 * scale)[0]
    assert (d == 0).mean() > 0.9 and len(ties) < 1e-3 * len(d), (float((d == 0).mean()), len(ties))
    a_ref, a_mine = _quad_area(g["mar_boxes"][ties]), _quad_area(boxes[ties])
    assert np.all(np.abs(a_ref - a_mine) <= 1e-6 * np.maximum(a_ref, 1e-12))


def test_convex_iou_oracle_bit_identical_to_reference_device_code(po):
    """SURVEY 8 n2: the reference's OWN devrIoU (convex_iou_kernel.cu:268-294, compiled as host C++) on 1000 x 40 pairs
    incl. duplicated points: the restatement reproduces every float bit for bit"""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "device_ops_ref.npz"))
    out = po.convex_iou(g["cx_pts"], g["cx_quads"])
    assert np.array_equal(out.view(np.uint32), g["cx_iou"].view(np.uint32))
    assert (g["cx_iou"] > 0.05).mean() > 0.05


def test_poly_nms_and_poly_overlaps_oracles_bit_identical_to_reference_device_code(po):
    """SURVEY 8 a15: DOTA_devkit/poly_nms_gpu has CUDA sources only; their __device__ functions compiled as host C++
    (oracle/build_ref.py) give tests/golden/device_ops_ref.npz.  The restatements reproduce every float: devPolyIoU of
    poly_nms_kernel.cu on 4000 clustered quad pairs, RotBox2Poly and devPolyIoU of poly_overlaps_kernel.cu on 300 x 40
    (cx, cy, w, h, theta) boxes."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "device_ops_ref.npz"))
    mine = np.array([po.iou_polynms_f32_one(p, q) for p, q in zip(g["pn_p"], g["pn_q"])], dtype=np.float32)
    assert np.array_equal(mine.view(np.uint32), g["pn_iou"].view(np.uint32))
    assert np.array_equal(po.rotbox_to_quad_f32(g["po_boxes"]), g["po_quads"])
    ov = po.poly_overlaps_f32(g["po_boxes"], g["po_query"])
    assert np.array_equal(ov.view(np.uint32), g["po_iou"].view(np.uint32)) and (ov > 0).mean() > 0.1


@pytest.mark.parametrize("case", [0, 1, 2, 3])
def test_dcn_oracle_vs_reference_im2col_kernels(case):
    """SURVEY 8 a6: tests/golden/device_ops_ref.npz holds weight x columns (the GEMM of deform_conv_cuda.cpp:231-236) over
    the column matrices the reference's OWN deformable_im2col_gpu_kernel / modulated_deformable_im2col_gpu_kernel
    (deform_conv_cuda_kernel.cu:190-243, :570-633) produce when their text is compiled as host C++ (float64; stride /
    padding / dilation variants, offsets leaving the image, DCNv2 mask).  It equals the oracle's deform_conv_ref."""
    import torch
    from oracle import torch_reference as tr
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "device_ops_ref.npz"))
    s_, p_, d_ = [int(v) for v in g["dcn%d_cfg" % case]]
    x, off, msk = (torch.from_numpy(g["dcn%d_%s" % (case, k)]) for k in ("x", "off", "mask"))
    wt = torch.from_numpy(g["dcn%d_w" % case])
    for key, mask in (("out", None), ("outm", msk)):
        ref = g["dcn%d_%s" % (case, key)]
        mine = tr.deform_conv_ref(x, off, wt, s_, p_, d_, mask=mask).numpy()
        assert mine.shape == ref.shape and np.abs(mine - ref).max() < 1e-12 * max(1.0, np.abs(ref).max())
