"""GPU: multi-scale tile producer (csrc/tiles.cu orp_resize_*; DESIGN.md §2 deviation 7) against the reference's own
splitter with the fixed-point contract as its resize (tests/golden/multiscale_tiles.json), the numpy restatement of the
contract (oracle/resize_cubic.py), the rate-1 producer, cv2, and the file-based ResultMerge."""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "multiscale_tiles.json")))


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch.device("cuda", 0)


def case_id(c):
    return "%dx%dx%d@%s" % (c["w"], c["h"], c["c"], c["rate"])


def rand_image(seed, h, w, c):
    return np.random.RandomState(seed).randint(0, 256, size=(h, w, c)).astype(np.uint8)


def all_tiles(img, name, rates, subsize, gap, batch=16, device=None):
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale
    tiles, names, origins = [], [], []
    for t, n, o in iter_tiles_multiscale(img, name, rates, subsize, gap, batch, device=device):
        tiles.append(t.clone())        # the producer reuses its batch buffers
        names += n
        origins += o
    return torch.cat(tiles), names, origins


@pytest.mark.parametrize("case", GOLD["cases"], ids=case_id)
def test_device_tiles_match_golden(cuda, case):
    img = rand_image(case["seed"], case["h"], case["w"], case["c"])
    tiles, names, _ = all_tiles(img, "P%04dx%04d" % (case["w"], case["h"]), (case["rate"],), GOLD["subsize"], GOLD["gap"],
                                device=cuda)
    assert names == [t[0] for t in case["tiles"]]
    host = tiles.cpu().numpy()
    for i, (name, sha) in enumerate(case["tiles"]):
        assert hashlib.sha1(np.ascontiguousarray(host[i]).tobytes()).hexdigest() == sha, name


def _device_table(n_src, rate, dev):
    from oracle import resize_cubic as rc
    from orientedreppoints_b200 import _lib
    n = rc.dst_size(n_src, rate)
    idx = torch.full((n, 4), -7, dtype=torch.int32, device=dev)
    w = torch.full((n, 4), -7, dtype=torch.int16, device=dev)
    _lib.check(_lib.lib().orp_resize_cubic_table(n_src, float(rate), n, _lib.ptr(idx), _lib.ptr(w), _lib.current_stream_ptr()),
               "orp_resize_cubic_table")
    return idx.cpu().numpy(), w.cpu().numpy()


@pytest.mark.parametrize("rate", [0.5, 0.75, 1.0, 1.25, 1.5, 2.0, 1 / 3, 0.1, 3.7, 0.999])
def test_device_tables_equal_oracle(cuda, rate):
    from oracle import resize_cubic as rc
    for n_src in (1, 2, 3, 5, 7, 10, 100, 517, 1021, 1024, 1025, 4000, 20000):
        if round(n_src * rate) < 1:
            continue
        idx, w = _device_table(n_src, rate, cuda)
        ri, rw = rc.table(n_src, rate)
        assert np.array_equal(idx, ri), (n_src, rate)
        assert np.array_equal(w, rw), (n_src, rate)


def test_full_image_equals_oracle(cuda):
    from oracle import resize_cubic as rc
    from orientedreppoints_b200.dota.split_tiles import resize_image_device
    rng = np.random.RandomState(2024)
    for k in range(20):
        w, h, c = int(rng.randint(1, 700)), int(rng.randint(1, 500)), int(rng.randint(1, 5))
        rate = float(rng.choice([0.5, 1.5, 0.75, 1.25, 2.0, rng.uniform(0.2, 2.5)]))
        if round(w * rate) < 1 or round(h * rate) < 1:
            continue
        img = rand_image(k, h, w, c)
        got = resize_image_device(torch.from_numpy(img).to(cuda), rate).cpu().numpy()
        assert np.array_equal(got, rc.resize(img, rate)), (w, h, c, rate)
    img = torch.from_numpy(rand_image(1, 30, 40, 3)).to(cuda)
    assert resize_image_device(img, 1.0) is img


def test_mixed_rate_batch_equals_per_rate_launches(cuda):
    from orientedreppoints_b200.dota.split_tiles import split_image
    img = rand_image(5, 900, 1300, 3)
    rates = (0.5, 1.0, 1.5, 0.75)
    mixed, names, origins = all_tiles(img, "P9", rates, 512, 128, batch=5, device=cuda)
    per_rate, per_names = [], []
    for r in rates:
        t, n, _ = all_tiles(img, "P9", (r,), 512, 128, batch=1000, device=cuda)
        per_rate.append(t)
        per_names += n
    assert names == per_names
    assert torch.equal(mixed, torch.cat(per_rate))
    ref, ref_names, ref_origins = split_image(img, "P9", 1.0, 512, 128, device=cuda)    # rate 1: the plain cut
    assert torch.equal(per_rate[1], ref)
    assert ref_names == [n for n in names if "__1.0__" in n]


def test_streaming_equals_all_at_once(cuda):
    img = rand_image(6, 2100, 1700, 3)
    a = all_tiles(img, "P3", (0.5, 1.0, 1.5), 1024, 200, batch=16, device=cuda)
    b = all_tiles(img, "P3", (0.5, 1.0, 1.5), 1024, 200, batch=10 ** 4, device=cuda)
    c = all_tiles(torch.from_numpy(img).to(cuda), "P3", (0.5, 1.0, 1.5), 1024, 200, batch=3, device=cuda)
    assert a[1] == b[1] == c[1] and a[2] == b[2] == c[2]
    assert torch.equal(a[0], b[0]) and torch.equal(a[0], c[0])


@pytest.mark.parametrize("rate", [0.5, 1.5])
def test_within_one_lsb_of_host_cv2_route(cuda, rate):
    pytest.importorskip("cv2")
    from orientedreppoints_b200.dota.split_tiles import split_image
    img = rand_image(7, 900, 1500, 3)
    dev, names, _ = all_tiles(img, "P5", (rate,), 1024, 200, device=cuda)
    host, host_names, _ = split_image(img, "P5", rate, 1024, 200, device=cuda)
    assert names == host_names
    assert (dev.int() - host.int()).abs().max().item() <= 1


def test_streaming_memory_is_image_plus_two_batches(cuda):
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale
    img = torch.randint(0, 256, (8000, 8000, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0)).numpy()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(cuda)
    probe = torch.empty(img.nbytes, dtype=torch.uint8, device=cuda)
    img_alloc = torch.cuda.memory_allocated(cuda) - base     # the image as the caching allocator holds it (2 MB granules)
    del probe
    torch.cuda.reset_peak_memory_stats(cuda)
    n = 0
    for tiles, names, _ in iter_tiles_multiscale(img, "P8", (0.5, 1.0, 1.5), 1024, 200, 16, device=cuda):
        n += tiles.shape[0]
    torch.cuda.synchronize()
    assert n == 25 + 100 + 225
    peak = torch.cuda.max_memory_allocated(cuda) - base
    assert peak <= img_alloc + 2 * 16 * 1024 * 1024 * 3 + (1 << 20), (peak, img_alloc)   # 432 MB if materialised at 1.5


def test_detect_image_multiscale_equals_file_based_merge(cuda, tmp_path):
    """streaming producer -> detector -> ONE merge over all rates == Task1 files of every rate through mergebypoly"""
    from orientedreppoints_b200.detector import OrientedRepPointsDetector
    from orientedreppoints_b200.dota import result_merge as rm
    from orientedreppoints_b200.dota.pipeline import DOTA_CLASSES, detect_image_multiscale, task1_lines
    from orientedreppoints_b200.weights import random_state_dict
    det = OrientedRepPointsDetector(random_state_dict(50, seed=0, reference_init=True), 50, cuda, "bf16",
                                    test_cfg=dict(score_thr=0.0, max_per_img=60))
    img = rand_image(11, 420, 610, 3)
    rates, kw = (0.5, 1.0, 1.5), dict(subsize=256, gap=64, batch=4)
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale
    # freeze the per-tile results (GroupNorm sums use atomics): both routes consume the same detections
    frozen, names, origins = [], [], []
    for t, n, o in iter_tiles_multiscale(img, "P0042", rates, kw["subsize"], kw["gap"], kw["batch"], device=cuda):
        frozen.append(det.simple_test(t))
        names += n
        origins += o
    res = [r for b in frozen for r in b]
    queue = list(frozen)

    def replay(t):
        out = queue.pop(0)
        assert len(out) == t.shape[0]
        return out
    det.simple_test = replay
    merged = detect_image_multiscale(det, img, "P0042", rates, merge_thresh=None, **kw)
    assert not queue and set(merged) == set(DOTA_CLASSES)
    assert {n.split("__")[1] for n in names} == {"0.5", "1.0", "1.5"}
    raw, out = tmp_path / "raw", tmp_path / "merged"
    rm.write_task1_raw(res, names, DOTA_CLASSES, str(raw))
    rm.mergebypoly(str(raw), str(out))
    total = 0
    for c in DOTA_CLASSES:
        lines = [l.rstrip("\n") for l in open(out / ("Task1_%s.txt" % c))]
        assert lines == merged[c], c
        total += len(lines)
    assert total > 0
    # a detection of a rate-1.5 tile comes back in image coordinates: (tile coordinate + tile origin) / 1.5
    per_class = task1_lines(res, names)
    line = next(l for lines in per_class for l in lines if "__1.5__" in l)
    sp = line.split(" ")
    k = names.index(sp[0])
    (l, u) = origins[k]
    _, _, dets = rm.parse_result_lines([line])
    poly = np.array(list(map(float, sp[2:10])))
    expect = (poly + np.tile([l, u], 4)) / 1.5
    assert np.allclose(dets[0, :8], expect, rtol=0, atol=1e-9) and dets[0, 8] == float(sp[1])


def test_bad_arguments_raise(cuda):
    from orientedreppoints_b200 import _lib
    from orientedreppoints_b200.dota.split_tiles import iter_tiles_multiscale, resize_image_device
    img = torch.zeros((64, 64, 3), dtype=torch.uint8, device=cuda)
    with pytest.raises(TypeError):
        resize_image_device(img.cpu(), 0.5)
    with pytest.raises(TypeError):
        resize_image_device(torch.zeros((64, 64, 5), dtype=torch.uint8, device=cuda), 0.5)
    with pytest.raises(ValueError):
        resize_image_device(img, 0.0)
    with pytest.raises(ValueError):
        resize_image_device(img, 0.001)
    with pytest.raises(ValueError):
        next(iter_tiles_multiscale(img, "P", rates=(0.5, -1.0)))
    l, st = _lib.lib(), _lib.current_stream_ptr()
    idx = torch.zeros((33, 4), dtype=torch.int32, device=cuda)
    w = torch.zeros((33, 4), dtype=torch.int16, device=cuda)
    assert l.orp_resize_cubic_table(64, 0.5, 31, _lib.ptr(idx), _lib.ptr(w), st) == -1          # n_dst != round(64 * 0.5)
    assert l.orp_resize_cubic_table(64, 0.0, 0, _lib.ptr(idx), _lib.ptr(w), st) == -1
    assert l.orp_resize_cubic_table(64, 0.5, 32, _lib.ptr(idx[0, 1:]), _lib.ptr(w), st) == -1   # misaligned
    rates = (ctypes.c_double * 9)(*([0.5] * 9))
    desc = torch.zeros((1, 3), dtype=torch.int32, device=cuda)
    out = torch.empty((1, 32, 32, 3), dtype=torch.uint8, device=cuda)
    args = (_lib.ptr(idx), _lib.ptr(w), _lib.ptr(idx), _lib.ptr(w), _lib.ptr(desc), 1, 32, _lib.ptr(out), st)
    assert l.orp_resize_tiles_cubic_u8(_lib.ptr(img), 64, 64, 5, 1, rates, *args) == -1           # C > 4
    assert l.orp_resize_tiles_cubic_u8(_lib.ptr(img), 64, 64, 3, 9, rates, *args) == -1           # too many rates
    assert l.orp_resize_tiles_cubic_u8(_lib.ptr(img), 64, 64, 3, 1, rates, None, None, None, None,
                                       _lib.ptr(desc), 1, 32, _lib.ptr(out), st) == -1             # rate 0.5 needs tables
    assert b"orp_resize_tiles_cubic_u8" in l.orp_last_error()
    assert l.orp_resize_cubic_u8(_lib.ptr(img), 64, 64, 3, 0.001, None, None, None, None, _lib.ptr(out), st) == -1
    torch.cuda.synchronize()
