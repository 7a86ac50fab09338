"""ctypes front-end of oracle/_build/liborp_oracle.so (TEST INFRASTRUCTURE ONLY).

Also holds the synthetic box generator of SURVEY.md section 8(d)-1 so tests, bench and the
golden-vector script share one definition.
"""
import ctypes
import os

import numpy as np

from . import build_oracle

_LIB = None
_REF = {}
HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")

c_dp = ctypes.POINTER(ctypes.c_double)
c_fp = ctypes.POINTER(ctypes.c_float)
c_ip = ctypes.POINTER(ctypes.c_int)


def lib():
    global _LIB
    if _LIB is None:
        path = build_oracle.build()
        _LIB = ctypes.CDLL(path)
        _LIB.orc_iou_poly_f64.restype = ctypes.c_double
        _LIB.orc_iou_rnms_f32.restype = ctypes.c_float
        _LIB.orc_iou_polynms_f32.restype = ctypes.c_float
    return _LIB


def _d(a):
    return a.ctypes.data_as(c_dp)


def _f(a):
    return a.ctypes.data_as(c_fp)


def _i(a):
    return a.ctypes.data_as(c_ip)


# ----------------------------------------------------------------------------- generators
def gen_rotated_boxes(n, seed=0, extent=1024.0, wmin=8.0, wmax=128.0):
    """SURVEY.md 8(d)-1 generator; lives in the product package (orientedreppoints_b200/synth.py) so that bench.py's
    product arm never imports oracle/"""
    from orientedreppoints_b200.synth import gen_rotated_boxes as g
    return g(n, seed, extent, wmin, wmax)


def gen_clustered_boxes(n_centres, copies, seed=0, extent=1024.0, jitter=4.0):
    """SURVEY.md B.5: object-like clusters (n_centres base boxes x `copies` jittered copies)."""
    base = gen_rotated_boxes(n_centres, seed=seed, extent=extent).astype(np.float64)
    rng = np.random.RandomState(seed + 1)
    reps = np.repeat(base, copies, axis=0)
    shift = rng.normal(0, jitter, (reps.shape[0], 1, 2))
    pts = reps[:, :8].reshape(-1, 4, 2) + shift + rng.normal(0, jitter * 0.25, (reps.shape[0], 4, 2))
    out = np.empty((reps.shape[0], 9), np.float32)
    out[:, :8] = pts.reshape(-1, 8).astype(np.float32)
    sc = np.sort(rng.uniform(0.05, 1.0, reps.shape[0]))[::-1].astype(np.float32)
    for k in range(1, sc.shape[0]):
        if sc[k] >= sc[k - 1]:
            sc[k] = np.nextafter(sc[k - 1], np.float32(-1))
    out[:, 8] = sc[rng.permutation(sc.shape[0])]
    return out


# ----------------------------------------------------------------------------- IoU
def iou_poly_f64(p, q):
    p = np.ascontiguousarray(p, np.float64).reshape(-1, 8)
    q = np.ascontiguousarray(q, np.float64).reshape(-1, 8)
    out = np.empty(p.shape[0], np.float64)
    lib().orc_iou_poly_f64_pairs(_d(p), _d(q), p.shape[0], _d(out))
    return out


def iou_rnms_f32(p, q):
    p = np.ascontiguousarray(p, np.float32).reshape(-1, 8)
    q = np.ascontiguousarray(q, np.float32).reshape(-1, 8)
    out = np.empty(p.shape[0], np.float32)
    lib().orc_iou_rnms_f32_pairs(_f(p), _f(q), p.shape[0], _f(out))
    return out


def iou_polynms_f32_one(p, q):
    p = np.ascontiguousarray(p, np.float32).reshape(8)
    q = np.ascontiguousarray(q, np.float32).reshape(8)
    return float(lib().orc_iou_polynms_f32(_f(p), _f(q)))


def iou_poly_f64_matrix(p, q):
    p = np.ascontiguousarray(p, np.float64).reshape(-1, 8)
    q = np.ascontiguousarray(q, np.float64).reshape(-1, 8)
    out = np.empty((p.shape[0], q.shape[0]), np.float64)
    lib().orc_iou_poly_f64_matrix(_d(p), p.shape[0], _d(q), q.shape[0], _d(out))
    return out


def rotbox_to_quad_f32(b):
    b = np.ascontiguousarray(b, np.float32).reshape(-1, 5)
    out = np.empty((b.shape[0], 8), np.float32)
    lib().orc_rotbox_to_quad_f32(_f(b), b.shape[0], _f(out))
    return out


def poly_overlaps_f32(b, q):
    b = np.ascontiguousarray(b, np.float32).reshape(-1, 5)
    q = np.ascontiguousarray(q, np.float32).reshape(-1, 5)
    out = np.empty((b.shape[0], q.shape[0]), np.float32)
    lib().orc_poly_overlaps_f32(_f(b), b.shape[0], _f(q), q.shape[0], _f(out))
    return out


# ----------------------------------------------------------------------------- NMS
def nms_poly_f64(dets, thresh, fast=False):
    """py_cpu_nms_poly / py_cpu_nms_poly_fast semantics; returns kept indices in score order."""
    d = np.ascontiguousarray(dets, np.float64).reshape(-1, 9)
    keep = np.empty(max(d.shape[0], 1), np.int32)
    fn = lib().orc_nms_poly_fast_f64 if fast else lib().orc_nms_poly_f64
    k = fn(_d(d), d.shape[0], ctypes.c_double(thresh), _i(keep))
    return keep[:k].copy()


def nms_f32(dets, thresh, guard=False):
    """rnms (guard=False) / poly_gpu_nms (guard=True) semantics; kept indices in score order."""
    d = np.ascontiguousarray(dets, np.float32).reshape(-1, 9)
    keep = np.empty(max(d.shape[0], 1), np.int32)
    k = lib().orc_nms_f32(_f(d), d.shape[0], ctypes.c_float(thresh), int(bool(guard)), _i(keep))
    return keep[:k].copy()


# ----------------------------------------------------------------------------- compiled reference
def ref_polyiou():
    if "poly" not in _REF:
        l = ctypes.CDLL(os.path.join(REF_DIR, "libref_polyiou.so"))
        l.ref_iou_poly.restype = ctypes.c_double
        _REF["poly"] = l
    return _REF["poly"]


def ref_iou_poly_pairs(p, q):
    p = np.ascontiguousarray(p, np.float64).reshape(-1, 8)
    q = np.ascontiguousarray(q, np.float64).reshape(-1, 8)
    out = np.empty(p.shape[0], np.float64)
    ref_polyiou().ref_iou_poly_pairs(_d(p), _d(q), p.shape[0], _d(out))
    return out


def ref_rnms():
    """reference rnms_cpu.cpp compiled unmodified (needs torch's shared libraries loaded)."""
    if "rnms" not in _REF:
        import torch  # noqa: F401  (loads libtorch so the extension's symbols resolve)
        l = ctypes.CDLL(os.path.join(REF_DIR, "ref_rnms_cpu.so"))
        l.ref_rotate_iou.restype = ctypes.c_float
        _REF["rnms"] = l
    return _REF["rnms"]


def ref_rotate_iou_pairs(p, q):
    p = np.ascontiguousarray(p, np.float32).reshape(-1, 8)
    q = np.ascontiguousarray(q, np.float32).reshape(-1, 8)
    out = np.empty(p.shape[0], np.float32)
    ref_rnms().ref_rotate_iou_pairs(_f(p), _f(q), p.shape[0], _f(out))
    return out


# ----------------------------------------------------------------------------- minarearect
def minarearect(pts18):
    """minaerarect oracle: float32 [n,18] (x0,y0..x8,y8) -> (boxes [n,8], hull_map [n,9], hull_n [n])."""
    p = np.ascontiguousarray(pts18, np.float32).reshape(-1, 18)
    n = p.shape[0]
    out = np.zeros((n, 8), np.float32)
    hmap = np.full((n, 9), -1, np.int32)
    hn = np.zeros(n, np.int32)
    lib().orc_minarearect(_f(p), n, _f(out), _i(hmap), _i(hn))
    return out, hmap, hn


def convex_iou(pts18, quads8):
    """IoU(hull of 9 points, quadrilateral) for every (point set, quad) pair: [N,18] x [K,8] -> float32 [N,K]
    (restated mmdet/ops/iou/src/convex_iou_kernel.cu:268-312)"""
    p = np.ascontiguousarray(pts18, dtype=np.float32).reshape(-1, 18)
    q = np.ascontiguousarray(quads8, dtype=np.float32).reshape(-1, 8)
    out = np.empty((p.shape[0], q.shape[0]), dtype=np.float32)
    lib().orc_convex_iou(p.ctypes.data_as(ctypes.c_void_p), p.shape[0], q.ctypes.data_as(ctypes.c_void_p), q.shape[0],
                         out.ctypes.data_as(ctypes.c_void_p))
    return out


def convex_hull9(pts18):
    p = np.ascontiguousarray(pts18, dtype=np.float32).reshape(18)
    ring = np.zeros(18, dtype=np.float64)
    n = lib().orc_convex_hull9(p.ctypes.data_as(ctypes.c_void_p), ring.ctypes.data_as(ctypes.c_void_p))
    return ring[:2 * n].reshape(-1, 2)
