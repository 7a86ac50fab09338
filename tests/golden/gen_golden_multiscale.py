"""Golden vectors for the multi-scale tile producer (DESIGN.md §2 deviation 7): runs the REFERENCE's own
splitbase.SplitSingle (DOTA_devkit/SplitOnlyImage_multi_process.py:51-87) with cv2.imread / cv2.imwrite replaced by
recorders and cv2.resize replaced by oracle/resize_cubic.py.  Tile names, origins, the zero padding and the rate-1
shortcut therefore come from the reference, the pixels from the fixed-point contract.  Per case it also records how far
the contract is from the installed cv2.resize(INTER_CUBIC), with the IPP HAL on and off (for the record only).

    python tests/golden/gen_golden_multiscale.py   # needs the reference's DOTA_devkit; writes tests/golden/multiscale_tiles.json
"""
import hashlib
import json
import os
import sys
import types

import numpy as np

REF = "/root/reference/DOTA_devkit"
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SPLIT_SIZES = [(1024, 1024), (1500, 900), (2048, 2048), (4000, 3000), (700, 500), (1024, 1025), (1849, 1848), (2672, 1024)]


def cases():
    """(w, h, c, rate): the split_tiles.json sizes at four rates, images whose scaled size drops below the 4-tap kernel
    or the tile, sizes whose scaled size is a .5 rounded to even, and one single-channel image"""
    out = [(w, h, 3, r) for (w, h) in SPLIT_SIZES for r in (0.5, 1.0, 1.5, 0.75)]
    out += [(7, 5, 3, 0.5), (7, 5, 3, 1.5), (7, 5, 3, 0.75), (1, 1, 3, 1.5), (1, 1, 3, 1.0), (3, 2, 3, 0.75)]
    out += [(1025, 1023, 3, 0.5), (1025, 1023, 3, 1.5), (1021, 517, 3, 0.5), (1021, 517, 3, 1.5)]
    out += [(1500, 900, 1, 0.5), (1500, 900, 1, 1.5)]
    return out


def image(w, h, c):
    seed = w * 7 + h + (c != 3)
    return seed, np.random.RandomState(seed).randint(0, 256, size=(h, w, c)).astype(np.uint8)


def cv2_distance(cv2, img, rate, ours):
    """(max |diff|, number of differing values) of cv2.resize against the contract, IPP HAL on and off"""
    out = {}
    was = cv2.ipp.useIPP()
    try:
        for key, ipp in (("ipp_on", True), ("ipp_off", False)):
            cv2.ipp.setUseIPP(ipp)
            ref = cv2.resize(img, None, fx=rate, fy=rate, interpolation=cv2.INTER_CUBIC).reshape(ours.shape)
            d = np.abs(ref.astype(np.int16) - ours.astype(np.int16))
            out[key] = [int(d.max()), int((d != 0).sum())]
    finally:
        cv2.ipp.setUseIPP(was)
    out["values"] = int(ours.size)
    return out


def main():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, REF)
    sys.modules.setdefault("dota_utils", types.ModuleType("dota_utils"))   # SplitSingle never touches it
    import cv2
    import SplitOnlyImage_multi_process as S
    from oracle import resize_cubic as rc

    out = {"gap": 200, "subsize": 1024, "cv2": cv2.__version__, "cases": []}
    for (w, h, c, rate) in cases():
        seed, img = image(w, h, c)
        rec = []
        sb = S.splitbase.__new__(S.splitbase)
        sb.srcpath = sb.dstpath = sb.outpath = "/nonexistent"
        sb.gap, sb.subsize, sb.slide, sb.ext, sb.padding = 200, 1024, 824, ".png", True
        orig = cv2.imread, cv2.imwrite, cv2.resize

        def fake_resize(src, dsize, fx, fy, interpolation):
            assert dsize is None and fx == fy and interpolation == cv2.INTER_CUBIC
            return rc.resize(src, fx)

        # saveimagepatches pads into a 3-channel canvas (broadcasting a single channel): keep the image's own channels
        cv2.imread = lambda path: img
        cv2.imwrite = lambda path, arr: rec.append(
            (os.path.basename(path)[:-4], hashlib.sha1(np.ascontiguousarray(arr[:, :, :c]).astype(np.uint8).tobytes()).hexdigest()))
        cv2.resize = fake_resize
        try:
            sb.SplitSingle("P%04dx%04d" % (w, h), rate, ".png")
        finally:
            cv2.imread, cv2.imwrite, cv2.resize = orig
        scaled = rc.resize(img, rate)
        case = {"w": w, "h": h, "c": c, "rate": rate, "seed": seed, "shape": list(scaled.shape[:2]), "tiles": rec}
        if rate != 1:
            case["cv2_diff"] = cv2_distance(cv2, img, rate, scaled)
        out["cases"].append(case)
        print(w, h, c, rate, scaled.shape, len(rec), case.get("cv2_diff"))
    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "multiscale_tiles.json")
    with open(dst, "w") as f:
        json.dump(out, f)
    print("wrote", dst, sum(len(c["tiles"]) for c in out["cases"]), "tiles")


if __name__ == "__main__":
    main()
