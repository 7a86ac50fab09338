"""Golden vectors for the two CUDA-only geometry ops (SURVEY §8 a8, n2) from the reference's OWN device code:
oracle/build_ref.py compiles the __device__ functions of
    mmdet/ops/minarearect/src/minarearect_kernel.cu   (Findminbox :343-452, Jarvis_and_index :215-341)
    mmdet/ops/iou/src/convex_iou_kernel.cu            (devrIoU :268-294)
    mmdet/ops/dcn/src/deform_conv_cuda_kernel.cu      ((modulated_)deformable_im2col_gpu_kernel :190-243, :570-633)
    DOTA_devkit/poly_nms_gpu/poly_nms_kernel.cu       (devPolyIoU :192-212)
    DOTA_devkit/poly_nms_gpu/poly_overlaps_kernel.cu  (RotBox2Poly :280-297, devPolyIoU :300-328)
as host C++ (the text above the __global__ kernels, separately rounded arithmetic); this script runs them.

    python oracle/build_ref.py && python tests/golden/gen_golden_device_ops.py    # needs /root/reference
"""
import ctypes
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po                                                    # noqa: E402


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def main():
    rm = ctypes.CDLL(os.path.join(ROOT, "oracle/_ref/ref_minarearect_dev.so"))
    rc = ctypes.CDLL(os.path.join(ROOT, "oracle/_ref/ref_convex_iou_dev.so"))
    rng = np.random.RandomState(0)
    n = 6000
    pts = rng.normal(0, 2.0, (n, 18)).astype(np.float32)
    pts[:200, 6:] = np.tile(pts[:200, :2], (1, 6))                                  # duplicated points
    g = np.stack(np.meshgrid(np.arange(3), np.arange(3)), -1).reshape(-1).astype(np.float32)
    pts[200:300] = g[None] * rng.randint(1, 5, (100, 1)).astype(np.float32) + rng.randint(-5, 5, (100, 1)).astype(np.float32)
    pts[300:400, 4:6] = (pts[300:400, 0:2] + pts[300:400, 2:4]) / 2                 # collinear triples
    boxes = np.zeros((n, 8), np.float32)
    rm.ref_minarearect(P(pts), n, P(boxes))
    maps = np.full((n, 9), -1, np.int32)
    hull_n = np.zeros(n, np.int32)
    for i in range(n):
        hull_n[i] = rm.ref_hull_index_map(P(pts[i]), P(maps[i]))
    N, K = 1500, 40
    p2 = (rng.rand(N, 9, 2) * 60 + rng.rand(N, 1, 2) * 100).astype(np.float32).reshape(N, 18)
    p2[:100, 6:] = np.tile(p2[:100, :2], (1, 6))
    q = po.gen_rotated_boxes(K, seed=4, extent=160.0, wmin=10, wmax=80)[:, :8].astype(np.float32)
    iou = np.zeros((N, K), np.float32)
    rc.ref_convex_iou(P(p2), N, P(q), K, P(iou))
    # DOTA_devkit/poly_nms_gpu: poly_nms_kernel.cu devPolyIoU (:192-212) on aligned quad pairs, poly_overlaps_kernel.cu
    # devPolyIoU / RotBox2Poly (:280-328) on (cx, cy, w, h, theta) boxes
    rn = ctypes.CDLL(os.path.join(ROOT, "oracle/_ref/ref_poly_nms_dev.so"))
    ro = ctypes.CDLL(os.path.join(ROOT, "oracle/_ref/ref_poly_overlaps_dev.so"))
    d = po.gen_clustered_boxes(60, 20, seed=5)
    r2 = np.random.RandomState(1)
    ii, jj = r2.randint(0, d.shape[0], 20000), r2.randint(0, d.shape[0], 20000)
    pp = np.ascontiguousarray(d[ii, :8], dtype=np.float32)
    qq = np.ascontiguousarray(d[jj, :8], dtype=np.float32)
    pn = np.zeros(20000, np.float32)
    rn.ref_poly_nms_iou_pairs(P(pp), P(qq), 20000, P(pn))
    b = np.stack([r2.uniform(0, 200, 300), r2.uniform(0, 200, 300), r2.uniform(5, 60, 300), r2.uniform(5, 60, 300),
                  r2.uniform(-3.2, 3.2, 300)], 1).astype(np.float32)
    qb = b[:40].copy()
    qb[:, :2] += r2.normal(0, 5, (40, 2)).astype(np.float32)
    ov = np.zeros((300, 40), np.float32)
    ro.ref_poly_overlaps(P(b), 300, P(qb), 40, P(ov))
    quads = np.zeros((300, 8), np.float32)
    ro.ref_rotbox2poly(P(b), 300, P(quads))
    # mmdet/ops/dcn/src/deform_conv_cuda_kernel.cu: (modulated_)deformable_im2col_gpu_kernel run on the host, float64
    rd = ctypes.CDLL(os.path.join(ROOT, "oracle/_ref/ref_dcn_dev.so"))
    dcn = {}
    r3 = np.random.RandomState(7)
    for ci, (nb, c, h, w, s_, p_, d_) in enumerate([(2, 8, 11, 13, 1, 1, 1), (1, 16, 9, 9, 2, 1, 1), (1, 4, 10, 12, 1, 2, 2), (3, 8, 7, 8, 1, 0, 1)]):
        ho, wo = (h + 2 * p_ - 2 * d_ - 1) // s_ + 1, (w + 2 * p_ - 2 * d_ - 1) // s_ + 1
        x = r3.randn(nb, c, h, w)
        off = r3.randn(nb, 18, ho, wo) * 2.5                                        # many samples leave the image
        msk = r3.rand(nb, 9, ho, wo)
        col1, col2 = np.zeros((c * 9, nb, ho, wo)), np.zeros((c * 9, nb, ho, wo))
        rd.ref_deformable_im2col_f64(P(x), P(off), None, nb, c, h, w, 3, 3, p_, s_, d_, P(col1))
        rd.ref_deformable_im2col_f64(P(x), P(off), P(msk), nb, c, h, w, 3, 3, p_, s_, d_, P(col2))
        # the convolution the columns feed (the GEMM of deform_conv_cuda.cpp:231-236) with 5 output channels
        wt = torch.randn(5, c, 3, 3, generator=torch.Generator().manual_seed(ci), dtype=torch.float64).numpy()
        conv = lambda col: (wt.reshape(5, c * 9) @ col.reshape(c * 9, -1)).reshape(5, nb, ho, wo).transpose(1, 0, 2, 3)  # noqa: E731
        dcn.update({"dcn%d_cfg" % ci: np.array([s_, p_, d_]), "dcn%d_x" % ci: x, "dcn%d_off" % ci: off, "dcn%d_mask" % ci: msk,
                    "dcn%d_w" % ci: wt, "dcn%d_out" % ci: conv(col1), "dcn%d_outm" % ci: conv(col2)})
    # stored: the first 4000 point sets, 1000 x 40 convex-IoU pairs and 4000 poly_nms pairs (every constructed special case
    # is among them), which keeps the file under 1 MB
    m, k = 4000, 1000
    np.savez_compressed(os.path.join(HERE, "device_ops_ref.npz"), **dcn, mar_pts=pts[:m], mar_boxes=boxes[:m], mar_map=maps[:m],
                        mar_hull_n=hull_n[:m], cx_pts=p2[:k], cx_quads=q, cx_iou=iou[:k], pn_p=pp[:m], pn_q=qq[:m], pn_iou=pn[:m],
                        po_boxes=b, po_query=qb, po_iou=ov, po_quads=quads)
    print("wrote device_ops_ref.npz", boxes.shape, iou.shape)


if __name__ == "__main__":
    main()
