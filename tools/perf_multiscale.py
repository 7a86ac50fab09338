"""Multi-scale tile producer measurements (DESIGN.md §4.3), one run on one GPU:

1. producer alone: CUDA events around one 16-tile batch at rate 1.5 cut from a 4000x4000x3 image
   (orp_resize_tiles_cubic_u8), against orp_split_tiles_u8 cutting the same 16 windows out of the image already resized
   to 6000x6000 (the copy roof of this shape).  L2 is overwritten (a 512 MB memset) before every timed launch.
2. the 16-tile R-50 f16x3 detector step, for scale.
3. end to end, one 4000x4000 image at rates (0.5, 1.0, 1.5), wall time ending in a synchronise:
   host route  = cv2 resize + split_image per rate, the detector, one merge over all rates;
   device route = detect_image_multiscale.

    python tools/perf_multiscale.py [--out results/perf_multiscale.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from orientedreppoints_b200 import _lib  # noqa: E402
from orientedreppoints_b200.dota import split_tiles as st  # noqa: E402
from orientedreppoints_b200.dota.pipeline import DOTA_CLASSES, detect_image_multiscale, task1_lines  # noqa: E402
from orientedreppoints_b200.dota.result_merge import merge_lines  # noqa: E402

HBM_PEAK = 7.7e12     # B200 data sheet, bytes/s


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def event_times(fn, reps, flush):
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), float(np.min(ts))


def producer(dev, reps):
    W = H = 4000
    rate, n, S = 1.5, 16, 1024
    img_h = np.random.RandomState(0).randint(0, 256, size=(H, W, 3)).astype(np.uint8)
    img = torch.from_numpy(img_h).to(dev)
    wr, hr = st.scaled_size(W, H, rate)
    org = st.tile_origins(wr, hr, S, 200)[:n]          # the first vertical strip, reference order
    xidx, xw, yidx, yw = st.resize_tables(W, H, [rate], dev)
    desc = torch.tensor([(0, l, u) for l, u in org], dtype=torch.int32, device=dev)
    out = torch.empty((n, S, S, 3), dtype=torch.uint8, device=dev)
    rates_c = (ctypes.c_double * 1)(rate)
    stream = _lib.current_stream_ptr()

    def resize_cut():
        _lib.check(_lib.lib().orp_resize_tiles_cubic_u8(_lib.ptr(img), H, W, 3, 1, rates_c, _lib.ptr(xidx), _lib.ptr(xw),
                                                        _lib.ptr(yidx), _lib.ptr(yw), _lib.ptr(desc), n, S, _lib.ptr(out),
                                                        stream), "resize")
    big = st.resize_image_device(img, rate)             # 6000x6000x3, the materialised image of the host route
    org_t = torch.tensor(org, dtype=torch.int32, device=dev)
    out2 = torch.empty_like(out)

    def plain_cut():
        _lib.check(_lib.lib().orp_split_tiles_u8(_lib.ptr(big), hr, wr, 3, _lib.ptr(org_t), n, S, _lib.ptr(out2), stream),
                   "split")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        resize_cut(), plain_cut()
    torch.cuda.synchronize()
    assert torch.equal(out, out2), "fused producer != resize + cut"
    bytes_out = n * S * S * 3
    res = {"shape": "16 tiles 1024x1024x3 at rate 1.5 from 4000x4000x3", "bytes_written": bytes_out, "l2": "flushed (512 MB memset) before every launch"}
    for name, fn in (("resize_tiles_cubic", resize_cut), ("split_tiles_copy_roof", plain_cut)):
        med, mn = event_times(fn, reps, flush)
        res[name] = {"ms_median": med, "ms_min": mn, "GBps_written": bytes_out / med / 1e6,
                     "share_of_7.7TBps": bytes_out / med / 1e-3 / HBM_PEAK}
    # the batch the producer writes runs through the detector next
    return res, out


def detector(dev):
    from orientedreppoints_b200.detector import OrientedRepPointsDetector
    from orientedreppoints_b200.weights import random_state_dict
    return OrientedRepPointsDetector(random_state_dict(50, seed=0, reference_init=True), 50, dev, "f16x3")


def detector_step(det, tiles, reps):
    for _ in range(2):
        det.simple_test(tiles)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        det.simple_test(tiles)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3


def host_route(det, img, name, rates, batch=16):
    results, names = [], []
    for r in rates:
        tiles, tn, _ = st.split_image(img, name, r, 1024, 200, device=det.device)
        for i in range(0, tiles.shape[0], batch):
            results.extend(det.simple_test(tiles[i:i + batch]))
        names += tn
    per_class = task1_lines(results, names)
    return {c: merge_lines(lines) for c, lines in zip(DOTA_CLASSES, per_class)}


def end_to_end(det, reps):
    import cv2
    img = np.random.RandomState(1).randint(0, 256, size=(4000, 4000, 3)).astype(np.uint8)
    rates = (0.5, 1.0, 1.5)
    routes = {"host_cv2": lambda: host_route(det, img, "P0001", rates),
              "device_fused": lambda: detect_image_multiscale(det, img, "P0001", rates)}
    for fn in routes.values():
        fn()
    ts = {k: [] for k in routes}
    outs = {}
    for _ in range(reps):                 # alternate the routes
        for k, fn in routes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[k] = fn()
            torch.cuda.synchronize()
            ts[k].append(time.perf_counter() - t0)
    t = time.perf_counter()
    for r in rates:
        st.resize_image(img, r)
    host_resize_ms = (time.perf_counter() - t) * 1e3
    ntiles = sum(len(st.tile_origins(*st.scaled_size(4000, 4000, r))) for r in rates)
    ndet = {k: sum(len(v) for v in o.values()) for k, o in outs.items()}
    return {"image": "4000x4000x3 at rates (0.5, 1.0, 1.5)", "tiles": ntiles, "cv2": cv2.__version__,
            "cv2_use_ipp": bool(cv2.ipp.useIPP()), "host_threads": os.cpu_count(),
            "host_cv2_resize_ms_all_rates": host_resize_ms,
            "ms_median": {k: float(np.median(v)) * 1e3 for k, v in ts.items()},
            "ms_all": {k: [x * 1e3 for x in v] for k, v in ts.items()}, "merged_detections": ndet}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--e2e-reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perf_multiscale.py measures on a GPU; none is present")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"card": card()}
    res["producer"], tiles = producer(dev, args.reps)
    print(json.dumps(res, indent=1), flush=True)
    det = detector(dev)
    step = detector_step(det, tiles, 10)
    res["detector_16_tiles_ms"] = step
    res["producer_share_of_detector_step"] = res["producer"]["resize_tiles_cubic"]["ms_median"] / step
    res["end_to_end"] = end_to_end(det, args.e2e_reps)
    print(json.dumps(res, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
