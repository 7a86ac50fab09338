"""Multi-scale tile producer, host side: the fixed-point INTER_CUBIC contract (DESIGN.md §2 deviation 7, restated in
oracle/resize_cubic.py) against the reference's own splitter run at rates != 1 (tests/golden/gen_golden_multiscale.py),
the size rule, the tile names, and the distance to cv2.resize where cv2 is installed."""
import hashlib
import json
import os

import numpy as np
import pytest

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "multiscale_tiles.json")))


def case_id(c):
    return "%dx%dx%d@%s" % (c["w"], c["h"], c["c"], c["rate"])


def golden_image(case):
    return np.random.RandomState(case["seed"]).randint(0, 256, size=(case["h"], case["w"], case["c"])).astype(np.uint8)


def cut(img, left, up, subsize):
    tile = np.zeros((subsize, subsize, img.shape[2]), np.uint8)
    part = img[up:up + subsize, left:left + subsize]
    tile[:part.shape[0], :part.shape[1]] = part
    return tile


@pytest.mark.parametrize("case", GOLD["cases"], ids=case_id)
def test_oracle_reproduces_reference_split(case):
    from oracle import resize_cubic as rc
    from orientedreppoints_b200.dota.split_tiles import tile_origins
    scaled = rc.resize(golden_image(case), case["rate"])
    assert list(scaled.shape[:2]) == case["shape"]
    org = tile_origins(scaled.shape[1], scaled.shape[0], GOLD["subsize"], GOLD["gap"])
    assert len(org) == len(case["tiles"])
    for (l, u), (name, sha) in zip(org, case["tiles"]):
        assert hashlib.sha1(cut(scaled, l, u, GOLD["subsize"]).tobytes()).hexdigest() == sha, name


@pytest.mark.parametrize("case", GOLD["cases"], ids=case_id)
def test_names_and_size_rule_match_reference(case):
    from oracle import resize_cubic as rc
    from orientedreppoints_b200.dota.split_tiles import scaled_size, tile_names, tile_origins
    wr, hr = scaled_size(case["w"], case["h"], case["rate"])
    assert [hr, wr] == case["shape"]
    assert (rc.dst_size(case["w"], case["rate"]), rc.dst_size(case["h"], case["rate"])) == (wr, hr)
    names = tile_names("P%04dx%04d" % (case["w"], case["h"]), case["rate"], tile_origins(wr, hr, GOLD["subsize"], GOLD["gap"]))
    assert names == [t[0] for t in case["tiles"]]
    assert all("__%s__" % case["rate"] in n for n in names)


def test_rate_is_printed_as_python_prints_it():
    from orientedreppoints_b200.dota.split_tiles import tile_names
    assert tile_names("P1", 1.0, [(0, 0)]) == ["P1__1.0__0___0"]
    assert tile_names("P1", 1, [(0, 0)]) == ["P1__1__0___0"]
    assert any(t[0].startswith("P1024x1024__1.0__") for c in GOLD["cases"] for t in c["tiles"])


def test_half_even_sizes():
    from orientedreppoints_b200.dota.split_tiles import scaled_size
    assert scaled_size(1025, 1023, 1.5) == (1538, 1534)
    assert scaled_size(1021, 517, 0.5) == (510, 258)
    assert scaled_size(5, 7, 0.5) == (2, 4)
    assert scaled_size(7, 5, 1.0) == (7, 5)


def test_tables_are_cv2_interpolate_cubic():
    """spot values: rate 1 is the identity tap, rate 0.5 samples half way between two pixels, taps replicate the border"""
    from oracle import resize_cubic as rc
    idx, w = rc.table(10, 1.0)
    assert (w == [0, 2048, 0, 0]).all() and (idx[:, 1] == np.arange(10)).all()
    idx, w = rc.table(8, 0.5)
    assert idx.tolist()[0] == [0, 0, 1, 2] and idx.tolist()[-1] == [5, 6, 7, 7]
    assert w.tolist()[1] == [-192, 1216, 1216, -192]     # interpolateCubic(0.5) * 2048


@pytest.mark.parametrize("rate", [0, -1.5, float("nan")])
def test_bad_rate_raises(rate):
    from oracle import resize_cubic as rc
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale, scaled_size
    with pytest.raises(ValueError):
        scaled_size(100, 100, rate)
    with pytest.raises(ValueError):
        rc.dst_size(100, rate)
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(np.zeros((100, 100, 3), np.uint8), "P", rates=(1.0, rate)))


def test_empty_result_raises():
    from oracle import resize_cubic as rc
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale, scaled_size
    for (w, h, r) in [(1, 1, 0.5), (10, 10, 0.04), (1000, 1, 0.2)]:
        with pytest.raises(ValueError):
            scaled_size(w, h, r)
        with pytest.raises(ValueError):
            rc.resize(np.zeros((h, w, 3), np.uint8), r)
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(np.zeros((1, 1, 3), np.uint8), "P", rates=(0.5,)))


def test_bad_multiscale_arguments_raise():
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale
    img = np.zeros((64, 64, 3), np.uint8)
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(img, "P", rates=()))
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(img, "P", rates=[0.5] * 9))
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(img, "P", batch=0))
    with pytest.raises(TypeError):
        next(iter_tiles_multiscale(img.astype(np.float32), "P"))
    with pytest.raises(TypeError):
        next(iter_tiles_multiscale(np.zeros((64, 64, 5), np.uint8), "P"))


@pytest.mark.parametrize("w,h,c,rate", [(1500, 900, 3, 1.5), (1500, 900, 3, 0.75), (1025, 1023, 3, 0.5), (1021, 517, 1, 1.5),
                                        (7, 5, 3, 1.25)])
def test_oracle_within_one_lsb_of_cv2(w, h, c, rate):
    cv2 = pytest.importorskip("cv2")
    from oracle import resize_cubic as rc
    img = np.random.RandomState(w + h + c).randint(0, 256, size=(h, w, c)).astype(np.uint8)
    ours = rc.resize(img, rate).astype(np.int16)
    was = cv2.ipp.useIPP()
    try:
        cv2.ipp.setUseIPP(False)       # OpenCV's own code: the vectorised float path differs from the integer one rarely
        d = np.abs(cv2.resize(img, None, fx=rate, fy=rate, interpolation=cv2.INTER_CUBIC).reshape(ours.shape) - ours)
        assert d.max() <= 1 and (d != 0).sum() <= 1e-3 * d.size
        cv2.ipp.setUseIPP(True)        # the default build (IPP HAL where present)
        d = np.abs(cv2.resize(img, None, fx=rate, fy=rate, interpolation=cv2.INTER_CUBIC).reshape(ours.shape) - ours)
        assert d.max() <= 1
    finally:
        cv2.ipp.setUseIPP(was)
