"""Mint the golden vectors of tests/golden/*.npz from the REFERENCE ITSELF (authoring container only).

Everything here executes reference code compiled/loaded from /root/reference via oracle/build_ref.py:
  * fp64 IoU      : DOTA_devkit/polyiou.cpp through the C harness (libref_polyiou.so)
  * fp32 IoU      : mmdet/ops/nms/src/rnms_cpu.cpp::rotate_iou through the C harness
  * fp64 NMS      : the reference's own python functions py_cpu_nms_poly (DOTA_devkit/ResultMerge.py:18-41)
                    and py_cpu_nms_poly_fast (ResultMerge_multi_process.py:60-121), extracted from the
                    reference files with `ast` (the modules themselves import unavailable packages)
                    and executed against the reference's SWIG module _polyiou
  * fp32 NMS      : rnms_cpu.soft_rnms(method=0) (the compiled torch extension)
The GPU box has no /root/reference: tests there only read the committed .npz files.

    python tests/golden/gen_golden.py
"""
import ast
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import build_ref, pyoracle as po  # noqa: E402

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


def _extract_function(path, name, namespace):
    src = open(path).read()
    tree = ast.parse(src)
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, path, "exec"), namespace)
            return namespace[name]
    raise KeyError(name)


def _load_ext(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def overlapping_pairs(dets, rng, n_pairs):
    """pairs whose AABBs overlap + jittered near-copies + a few analytic cases"""
    q = dets[:, :8].astype(np.float64)
    x1, x2 = q[:, 0::2].min(1), q[:, 0::2].max(1)
    y1, y2 = q[:, 1::2].min(1), q[:, 1::2].max(1)
    ii, jj = [], []
    n = len(dets)
    for i in range(n):
        m = (x1 < x2[i]) & (x2 > x1[i]) & (y1 < y2[i]) & (y2 > y1[i])
        m[i] = False
        for j in np.nonzero(m)[0]:
            ii.append(i)
            jj.append(j)
    ii, jj = np.array(ii), np.array(jj)
    sel = rng.permutation(len(ii))[: n_pairs // 2]
    p = [dets[ii[sel], :8]]
    qq = [dets[jj[sel], :8]]
    # jittered copies (high IoU, nearly parallel edges)
    k = n_pairs // 2 - 16
    src = dets[rng.randint(0, n, k), :8].astype(np.float64)
    jit = src + rng.normal(0, 1.5, src.shape)
    p.append(src.astype(np.float32))
    qq.append(jit.astype(np.float32))
    # analytic cases
    sq = np.array([0, 0, 1, 0, 1, 1, 0, 1], np.float32)
    cases = [
        (sq, sq + 0.5),                                   # polyiou.cpp:130-136 -> 1/7
        (sq, sq),                                         # identical -> 1
        (sq, sq + 2.0),                                   # disjoint -> 0
        (sq, sq + np.array([1, 0] * 4, np.float32)),      # shared edge -> 0
        (sq, sq[::-1].reshape(4, 2)[:, ::-1].reshape(-1)),  # same square, clockwise order
        (sq * 100, sq * 10 + 20),                         # contained
        (sq * 100 + 500, (sq * 100 + 500)),               # identical far from origin
        (np.array([0, 0, 4, 0, 4, 2, 0, 2], np.float32), np.array([2, -1, 3, -1, 3, 3, 2, 3], np.float32)),  # cross
    ]
    c, s = np.cos(np.pi / 4), np.sin(np.pi / 4)
    rot = np.array([[c, -s], [s, c]])
    sq45 = ((sq.reshape(4, 2) - 0.5) @ rot.T + 0.5).reshape(-1).astype(np.float32)
    cases.append((sq, sq45))                              # 45 degree copy
    cases.append((sq * 1000 + 300, sq45 * 1000 + 300))
    while len(cases) < 16:
        cases.append((sq * (len(cases) + 1), sq * (len(cases) + 1) + 0.25 * len(cases)))
    p.append(np.stack([a for a, _ in cases]).astype(np.float32))
    qq.append(np.stack([b for _, b in cases]).astype(np.float32))
    return np.concatenate(p).astype(np.float32), np.concatenate(qq).astype(np.float32)


def clustered_pairs():
    """iou_clustered.npz: 4000 random pairs of object-like clusters (many near-duplicates) through polyiou.cpp (fp64) and
    rnms_cpu.cpp rotate_iou (fp32)"""
    d = po.gen_clustered_boxes(40, 12, seed=11)
    rng = np.random.RandomState(5)
    i, j = rng.randint(0, len(d), 4000).astype(np.int32), rng.randint(0, len(d), 4000).astype(np.int32)
    p, q = d[i, :8], d[j, :8]
    np.savez_compressed(os.path.join(OUT, "iou_clustered.npz"), dets=d, i=i, j=j,
                        ref64=po.ref_iou_poly_pairs(p, q), ref32=po.ref_rotate_iou_pairs(p, q))
    print("iou_clustered:", p.shape)


def main():
    assert os.path.isdir(REF), "golden vectors can only be minted where /root/reference exists"
    build_ref.build(verbose=True)
    sys.path.insert(0, po.REF_DIR)
    import polyiou as ref_polyiou_swig  # the reference's SWIG module
    import torch
    ref_rnms_mod = _load_ext("ref_rnms_cpu", os.path.join(po.REF_DIR, "ref_rnms_cpu.so"))

    ns = {"polyiou": ref_polyiou_swig, "np": np}
    py_cpu_nms_poly = _extract_function(os.path.join(REF, "DOTA_devkit/ResultMerge.py"), "py_cpu_nms_poly", ns)
    ns2 = {"polyiou": ref_polyiou_swig, "np": np, "math": __import__("math"), "pdb": __import__("pdb")}
    py_cpu_nms_poly_fast = _extract_function(os.path.join(REF, "DOTA_devkit/ResultMerge_multi_process.py"),
                                             "py_cpu_nms_poly_fast", ns2)

    rng = np.random.RandomState(1234)
    # ---------------------------------------------------------------- IoU pairs
    dets = po.gen_rotated_boxes(1000, seed=0)
    p, q = overlapping_pairs(dets, rng, 3000)
    ref64 = po.ref_iou_poly_pairs(p, q)
    ref32 = po.ref_rotate_iou_pairs(p, q)
    swig_check = np.array([ref_polyiou_swig.iou_poly(ref_polyiou_swig.VectorDouble([float(v) for v in a]),
                                                     ref_polyiou_swig.VectorDouble([float(v) for v in b]))
                           for a, b in zip(p[:200], q[:200])])
    assert np.array_equal(swig_check, ref64[:200], equal_nan=True)
    np.savez_compressed(os.path.join(OUT, "iou_pairs.npz"), p=p, q=q, ref64=ref64, ref32=ref32)
    print("iou_pairs:", p.shape, "nonzero", int((ref64 > 1e-9).sum()), "max|f32-f64|", float(np.nanmax(np.abs(ref32 - ref64))))
    clustered_pairs()

    # ---------------------------------------------------------------- NMS, config[0] of BASELINE.json
    def nms_suite(name, d):
        d64 = d.astype(np.float64)
        out = {"dets": d}
        for thr in (0.1, 0.3):
            out["keep64_thr%02d" % int(thr * 10)] = np.array(py_cpu_nms_poly(d64, thr), np.int64)
        out["keep64fast_thr01"] = np.array(py_cpu_nms_poly_fast(d64, 0.1), np.int64)
        for thr in (0.1, 0.4):
            r = ref_rnms_mod.soft_rnms(torch.from_numpy(d.copy()), float(thr), 0, 0.5, 1e-3)
            out["keep32_thr%02d" % int(thr * 10)] = r[:, 9].numpy().astype(np.int64)   # selection order
        np.savez_compressed(os.path.join(OUT, name), **out)
        print(name, {k: (v.shape if k == "dets" else len(v)) for k, v in out.items()})
        return out

    nms_suite("nms_1k.npz", dets)
    nms_suite("nms_clustered.npz", po.gen_clustered_boxes(60, 10, seed=3))
    # H1: the same boxes far from the origin (what the class-offset trick does)
    far = dets.copy()
    far[:, :8] += 16000.0
    nms_suite("nms_1k_offset16000.npz", far)


if __name__ == "__main__":
    main()
