"""Tile-throughput workload of bench.py: BASELINE.json configs[1] - R-50 + FPN + OrientedRepPointsHead on
synthetic 1024x1024 tiles, random-init weights, one process per GPU, tiles sharded across ranks (weak
scaling: `batch` tiles per GPU per step), ONE all-gather of the per-tile detections per step when N > 1.

score_thr is set to 0 (SURVEY.md H8): with random-init weights every sigmoid score is ~0.01 < 0.05 and the
config-faithful run would hand an empty set to NMS; with 0 every tile feeds 80 160 candidates to
multiclass_rnms, which is the load BASELINE.json describes ("~10^5 proposals per tile").
"""
import time

import numpy as np
import torch

from . import _lib
from .core.transforms import rbbox2result
from .detector import OrientedRepPointsDetector
from .weights import STAGE_BLOCKS, random_state_dict


def conv_flops_per_tile(depth=50, size=1024):
    """2*MACs of every convolution (dense or deformable) of the graph for one size x size tile."""
    fl = 0.0
    s = size // 2
    fl += 2.0 * s * s * 64 * 147                                       # conv1 7x7/2
    s //= 2                                                            # maxpool
    inpl = 64
    for li, (nblk, planes) in enumerate(zip(STAGE_BLOCKS[depth], (64, 128, 256, 512))):
        for b in range(nblk):
            st = 2 if (b == 0 and li > 0) else 1
            so = s // st
            fl += 2.0 * s * s * planes * inpl                          # conv1 1x1 (input resolution)
            fl += 2.0 * so * so * planes * planes * 9                  # conv2 3x3 (stride here: style='pytorch')
            fl += 2.0 * so * so * planes * 4 * planes                  # conv3 1x1
            if b == 0:
                fl += 2.0 * so * so * planes * 4 * inpl                # downsample
            inpl = planes * 4
            s = so
    lv = [size // 8, size // 16, size // 32, size // 64, size // 128]
    for hw, cin in zip(lv[:3], (512, 1024, 2048)):
        fl += 2.0 * hw * hw * 256 * cin                                # laterals
        fl += 2.0 * hw * hw * 256 * 256 * 9                            # fpn convs
    fl += 2.0 * lv[3] * lv[3] * 256 * 2048 * 9                         # P6 on C5
    fl += 2.0 * lv[4] * lv[4] * 256 * 256 * 9                          # P7
    loc = sum(h * h for h in lv)
    per_loc = 2.0 * (6 * 256 * 256 * 9 + 256 * 256 * 9 + 256 * 18 + 2 * 256 * 256 * 9 + 256 * 15 + 256 * 18)
    fl += loc * per_loc
    return fl


def swin_flops_per_tile(size=1024):
    """2*MACs of the Swin-T backbone (Linear layers + window attention on the 7-padded grids) + its FPN + the head."""
    fl = 0.0
    h = size // 4
    fl += 2.0 * h * h * 96 * 48                                        # patch embed
    for i, depth in enumerate((2, 2, 6, 2)):
        c = 96 << i
        hp = (h + 6) // 7 * 7
        for _ in range(depth):
            fl += 2.0 * hp * hp * 3 * c * c                            # qkv on the padded grid
            fl += 2.0 * hp * hp * 49 * c * 2                           # QK^T and PV
            fl += 2.0 * h * h * c * c                                  # proj
            fl += 2.0 * h * h * 8 * c * c                              # MLP
        if i < 3:
            fl += 2.0 * (h // 2) * (h // 2) * 4 * c * 2 * c            # patch merging reduction
            h //= 2
    lv = [size // 8, size // 16, size // 32, size // 64, size // 128]
    for hw, cin in zip(lv[:3], (192, 384, 768)):
        fl += 2.0 * hw * hw * 256 * cin + 2.0 * hw * hw * 256 * 256 * 9
    loc = sum(v * v for v in lv)
    fl += loc * 2.0 * (6 * 256 * 256 * 9 + 256 * 256 * 9 + 256 * 18 + 2 * 256 * 256 * 9 + 256 * 15 + 256 * 18)
    return fl


def build_detector(backbone, precision, dev, reference_init=True):
    if backbone == "swin_tiny":
        from .swin import random_swin_state_dict
        depth, sd = "swin_tiny", random_swin_state_dict(0)
    else:
        depth = int(backbone[1:])
        sd = random_state_dict(depth, seed=0, reference_init=reference_init)
    return depth, OrientedRepPointsDetector(sd, depth, dev, precision, test_cfg=dict(score_thr=0.0))


def _device_steps(det, img, steps, warm, world, flush, benchmod, use_graph, sampler=None):
    """`steps` device-resident steps (dense graph -> fused post-processing -> packed detections -> all-gather), CUDA events
    around every step, L2 flush between steps.  The collective is asynchronous: step s waits for the gather of step s-1
    (the last step also for its own), so the ranks are not forced into lockstep and the gather overlaps the next step's
    dense graph.  Returns (ms per step as max over ranks, per-tile detection counts, launches counted by the library,
    (dets, labels, counts) as simple_test returned them in the last step)."""
    from . import gather as G
    pending = [None]
    out = [None]

    def step(last=False):
        dets, labels, counts = out[0] = det.simple_test(img, return_tensors="padded")
        buf, _ = G.pack(dets, labels, counts)
        h = G.all_gather_detections(buf, async_op=True)
        res = pending[0].wait() if pending[0] is not None else None
        pending[0] = h
        if last:
            res = h.wait()
            pending[0] = None
        return res

    if use_graph:
        det.capture(img.shape, img.dtype)
    for i in range(warm):
        step(last=(i == warm - 1))
    benchmod.barrier(world)
    if sampler is not None:
        sampler.start()                                       # nvidia-smi clocks DURING the timed region
    _lib.reset_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    benchmod.barrier(world)
    all_cnt = None
    for s in range(steps):
        flush.fill_(s & 0xFF)
        ev[s][0].record()
        got = step(last=(s == steps - 1))                     # the last step drains its own gather inside the timed region
        ev[s][1].record()
        if got is not None:
            _, all_cnt = got
    benchmod.barrier(world)
    launches = _lib.launch_count()
    total_ms = benchmod.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev), world)
    return total_ms / steps, [int(v) for v in all_cnt.reshape(-1).tolist()], launches, out[0]


def step_outputs(dets, labels, counts, limit):
    """host copy of what simple_test returned in a step: the valid detections of every tile concatenated in tile order
    (float32 [sum(counts), 27], the rows the padded output holds), their labels, the per-tile counts and the tile indices.
    If every tile would take more than `limit` bytes, a fixed, seeded sample of the tiles is kept."""
    n, cap = dets.shape[0], dets.shape[1]
    per_tile = cap * (dets.shape[2] * 4 + 8) + 16
    tiles = np.arange(n)
    if n * per_tile > limit:
        tiles = np.sort(np.random.RandomState(0).choice(n, limit // per_tile, replace=False))
    cnt = counts.cpu().numpy()[tiles]
    valid = np.arange(cap)[None, :] < cnt[:, None]
    return {"detections": dets.cpu().numpy()[tiles][valid], "labels": labels.cpu().numpy()[tiles][valid],
            "counts": cnt, "tiles": tiles}


def _roofline_pass(det, img, steps, flush):
    """the same dense graph launched eagerly (a CUDA graph cannot carry per-launch events), every tensor-core convolution
    bracketed by CUDA events on its launching stream: (kernel ms per step, launches per step, algorithmic flops per step,
    all library launches of one eager dense pass)"""
    saved = getattr(det, "_g_shape", None)
    det._g_shape = None
    before = _lib.launch_count()
    det.forward_dense(img)
    launches_dense = _lib.launch_count() - before
    _lib.set_timing(True)
    _lib.tc_timing_collect()
    n = max(1, min(steps, 10))                                # the library keeps 1024 event pairs
    for s in range(n):
        flush.fill_(s & 0xFF)
        det.forward_dense(img)
    torch.cuda.synchronize()
    tc_ms, tc_launches, tc_flops = _lib.tc_timing_collect()
    _lib.set_timing(False)
    det._g_shape = saved
    return tc_ms / n, tc_launches // n, tc_flops / n, launches_dense


def _roofline_obj(precision, kernel_ms, tc_launches, flops_step, ms_step, pk, batch, fl_tile, traffic=None, traffic_note=None):
    """`achieved` = ALGORITHMIC flops (2*MACs of the convolutions, no padded / identity / extra-term MMAs) / kernel time.
    The f16x3 mode executes three MMAs per algorithmic product, so its tensor pipe is three times as busy as `frac` says:
    `tensor_pipe_frac` (executed MMA flops / peak) is the utilisation north_star's 70 % target speaks of."""
    ach = flops_step / (kernel_ms * 1e-3) / 1e12
    mult = 3.0 if precision == "f16x3" else 1.0
    return {"bound": "tensor", "kernel": "conv_tc_kernel (all %d launches per step)" % tc_launches,
            "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
            "mma_per_product": mult, "executed_tflops": ach * mult, "tensor_pipe_frac": ach * mult / pk["bf16_tflops_sustained"],
            "traffic": traffic, "traffic_note": traffic_note, "peak_source": pk["source"] + " (sustained, dense bf16/fp16)",
            "algorithmic_flops_per_step": flops_step, "kernel_ms_per_step": kernel_ms,
            "kernel_share_of_step": kernel_ms / ms_step,
            "whole_step_tflops": batch * fl_tile / (ms_step * 1e-3) / 1e12}


def detection_diff(det_a, det_b, img, tiles=2):
    """detection-level difference of two engines on the same tiles (score_thr 0, 2000 detections per tile): detections are
    matched by label and nearest box (8 coordinates, L-inf)"""
    out = []
    for det in (det_a, det_b):
        saved = getattr(det, "_g_shape", None)
        det._g_shape = None
        out.append(det.simple_test(img[:tiles].contiguous(), return_tensors="padded"))
        det._g_shape = saved
    (da, la, ca), (db, lb, cb) = out
    rep = {"tiles": tiles, "counts_a": ca.tolist(), "counts_b": cb.tolist(), "matched_within_1px": [], "matched_within_0p01px": [],
           "median_coord_delta_px": [], "max_score_delta_of_matched": []}
    for t in range(tiles):
        a, b = da[t, :int(ca[t])], db[t, :int(cb[t])]
        if a.shape[0] == 0 or b.shape[0] == 0:
            continue
        dist = torch.cdist(a[:, 18:26].double(), b[:, 18:26].double(), p=float("inf"))
        dist = dist + (la[t, :a.shape[0], None] != lb[t, None, :b.shape[0]]).double() * 1e6
        best, arg = dist.min(dim=1)
        rep["matched_within_1px"].append(float((best < 1.0).float().mean()))
        rep["matched_within_0p01px"].append(float((best < 0.01).float().mean()))
        rep["median_coord_delta_px"].append(float(best.median()))
        m = best < 1.0
        rep["max_score_delta_of_matched"].append(float((a[m, 26] - b[arg[m], 26]).abs().max()) if bool(m.any()) else None)
    return rep


def run_config(backbone, precision, batch, args, rank, world, local, benchmod, flush, steps=None, reference_init=True):
    """one extra configuration measured the same way (device-timed steps + roofline pass): used for BASELINE.json configs 4
    (R-101, 4 tiles/GPU) and 5 (Swin-T + DCN head, 8 tiles/GPU) and for the bf16 arithmetic of the headline config"""
    dev = torch.device("cuda", local)
    depth, det = build_detector(backbone, precision, dev, reference_init)
    g = torch.Generator().manual_seed(1000 + rank)
    img = torch.randint(0, 256, (batch, 1024, 1024, 3), generator=g, dtype=torch.uint8).to(dev)
    steps = steps or max(3, min(args.steps, 10))
    ms_step, ndet, _, _ = _device_steps(det, img, steps, 3, world, flush, benchmod, not getattr(args, "no_graph", False))
    pk = benchmod.peaks()
    fl_tile = swin_flops_per_tile() if depth == "swin_tiny" else conv_flops_per_tile(depth)
    k_ms, k_n, k_fl, _ = _roofline_pass(det, img, steps, flush)
    out = {"workload": "%s FPN OrientedRepPoints, %d synthetic 1024x1024 tiles per GPU per step, %s arithmetic"
                       % ("Swin-T" if depth == "swin_tiny" else "R-%d" % depth, batch, precision),
           "value": world * batch / (ms_step * 1e-3), "unit": "tiles/s", "n_gpus": world, "steps": steps, "ms_per_step": ms_step,
           "dtype": precision, "tiles_per_gpu_per_step": batch, "gflop_per_tile": fl_tile / 1e9, "detections_per_tile": ndet[:4],
           "roofline": _roofline_obj(precision, k_ms, k_n, k_fl, ms_step, pk, batch, fl_tile)}
    if hasattr(det.eng, "overflow_count"):
        out["f16_overflow_events"] = det.eng.overflow_count()
    return out, det, img


def run(args, rank, world, local, benchmod):
    dev = torch.device("cuda", local)
    batch = args.batch or 16     # tiles per GPU per step: 8 -> 16 amortises the fixed cost of the small late-backbone launches (+11 %)
    precision = args.precision or "f16x3"
    backbone = getattr(args, "backbone", None) or "r50"
    depth, det = build_detector(backbone, precision, dev)
    g = torch.Generator().manual_seed(1000 + rank)
    # decoded tiles as the data pipeline holds them: uint8 HWC; Normalize (mean/std/to_rgb) runs on the device
    img_host = torch.randint(0, 256, (batch, 1024, 1024, 3), generator=g, dtype=torch.uint8).pin_memory()
    img = img_host.to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    warm = max(args.warmup, 3)

    from . import gather as G

    use_graph = not getattr(args, "no_graph", False)
    sampler = benchmod.ClockSampler(local)
    ms_step, ndet, launches, last = _device_steps(det, img, args.steps, warm, world, flush, benchmod, use_graph,
                                                  sampler=sampler if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        benchmod.write_outputs(args.dump_outputs, step_outputs(*last, benchmod.DUMP_LIMIT))
    # roofline pass
    tc_ms, tc_launches, tc_flops, launches_dense = _roofline_pass(det, img, args.steps, flush)
    if use_graph:
        launches += args.steps * launches_dense                 # kernels inside the replayed graph are not seen by the library's counter
    # end to end through the public API: pinned host tiles -> H2D -> simple_test -> rbbox2result (D2H), every step.
    # The H2D copy of step i+1 is issued on a copy stream while step i computes (what a prefetching data loader
    # does); every step still moves its own input bytes host->device and its own detections device->host.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [torch.empty_like(img), torch.empty_like(img)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            bufs[slot].copy_(img_host, non_blocking=True)
            ready[slot].record(copy_stream)

    # Results come back through pinned host buffers; a step's D2H copy is queued right behind its kernels and is
    # collected (event wait + rbbox2result on the host) after the NEXT step's GPU work has been issued, so the host
    # never idles the GPU - the loop a serving process runs.
    cap = int(det.test_cfg["max_per_img"])
    host_out = [dict(d=torch.empty((batch, cap, 27), dtype=torch.float32).pin_memory(),
                     l=torch.empty((batch, cap), dtype=torch.int64).pin_memory(),
                     c=torch.empty((batch,), dtype=torch.int32).pin_memory(), ev=torch.cuda.Event()) for _ in range(2)]

    def issue_e2e(slot, prefetch_next):
        torch.cuda.current_stream().wait_event(ready[slot])
        if prefetch_next:
            upload(slot ^ 1)
        dets, labels, counts = det.simple_test(bufs[slot], return_tensors="padded")
        gh = G.all_gather_detections(G.pack(dets, labels, counts)[0], async_op=True)
        consumed[slot].record(torch.cuda.current_stream())
        h = host_out[slot]
        h["gather"] = gh
        h["d"].copy_(dets, non_blocking=True)                         # device -> host: the step's result
        h["l"].copy_(labels, non_blocking=True)
        h["c"].copy_(counts, non_blocking=True)
        h["ev"].record(torch.cuda.current_stream())
        return slot

    def collect_e2e(slot):
        h = host_out[slot]
        h["gather"].wait()                                            # every rank now holds every rank's detections
        h["ev"].synchronize()
        cnt = h["c"].tolist()
        return [rbbox2result(h["d"][i, :cnt[i]], h["l"][i, :cnt[i]], 16) for i in range(batch)]

    for c in consumed:
        c.record(torch.cuda.current_stream())
    upload(0)
    for i in range(2):
        collect_e2e(issue_e2e(i & 1, True))
    benchmod.barrier(world)
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    pending = None
    for i in range(e2e_steps):
        cur = issue_e2e(i & 1, i + 1 < e2e_steps)
        if pending is not None:
            out = collect_e2e(pending)
        pending = cur
    out = collect_e2e(pending)
    torch.cuda.synchronize()
    e2e_ms = benchmod.max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps, world)
    d2h = sum(int(host_out[0][k].nbytes) for k in ("d", "l", "c"))

    # BASELINE.json configs[1] names a SINGLE tile: the same path with one tile per step (latency-bound: the dense graph
    # is ~75 launches whatever the batch), reported next to the throughput configuration above
    single = None
    if use_graph and batch > 1:
        img1 = img[:1].contiguous()
        det.capture(img1.shape, img1.dtype)
        for _ in range(3):
            det.simple_test(img1, return_tensors="padded")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n1 = 20
        e0.record()
        for _ in range(n1):
            det.simple_test(img1, return_tensors="padded")
        e1.record()
        torch.cuda.synchronize()
        ms1 = benchmod.max_over_ranks(e0.elapsed_time(e1) / n1, world)
        single = {"tiles_per_gpu_per_step": 1, "ms_per_step": ms1, "value": world * 1.0 / (ms1 * 1e-3), "unit": "tiles/s",
                  "note": "device-timed, inputs resident, no L2 flush between steps"}

    pk = benchmod.peaks()
    fl_tile = swin_flops_per_tile() if depth == "swin_tiny" else conv_flops_per_tile(depth)
    line = {
        "metric": "1024x1024 tiles/sec", "value": world * batch / (ms_step * 1e-3), "unit": "tiles/s", "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": precision, "data": "synthetic",
        "config": {"workload": "%s FPN OrientedRepPoints, %d synthetic 1024x1024 tile(s) per GPU per step, random-init "
                               "weights, score_thr=0 (80160 NMS candidates per tile), rnms iou 0.4, max_per_img 2000"
                               % ("Swin-T" if depth == "swin_tiny" else "R-%d" % depth, batch),
                   "tiles_per_gpu_per_step": batch, "detections_per_tile": ndet[:4],
                   "l2": "512 MiB flush write between timed steps", "gflop_per_tile": fl_tile / 1e9,
                   "cuda_graph": "dense graph (backbone+FPN+head) replayed as one CUDA graph" if use_graph else "eager launches",
                   "gather": "one asynchronous all_gather_into_tensor of [tiles,2001,28] fp32 (detections + count row) per step" if world > 1 else "single rank"},
        "gpu_launches": int(launches),
        "single_tile_step": single,
        "e2e": {"value": world * batch / (e2e_ms * 1e-3), "unit": "tiles/s", "h2d_bytes_per_step": int(img_host.nbytes),
                "d2h_bytes_per_step": int(d2h), "api": "OrientedRepPointsDetector.simple_test(uint8 HWC tiles) -> rbbox2result lists", "input": "uint8 HWC tiles, Normalize fused into the stem input transform"},
    }
    traffic, traffic_note = None, None
    try:
        import json as _json
        import os as _os
        name = "r2_conv_tc_traffic_%s_b%d.json" % (precision, batch)
        tj = _json.load(open(_os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))), "profiles", name)))
        if depth == 50 and batch == tj["tiles"]:
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]      # ncu, all conv launches of one step (cold L2 per launch)
            traffic_note = "dram bytes read+written by the same launches under ncu (profiles/%s)" % name
    except Exception:
        pass
    if tc_ms > 0:
        line["roofline"] = _roofline_obj(precision, tc_ms, tc_launches, tc_flops, ms_step, pk, batch, fl_tile, traffic, traffic_note)
    if hasattr(det.eng, "overflow_count"):
        line["f16_overflow_events"] = det.eng.overflow_count()
    line["parity"] = ("f16x3: every fp32 product as fp16 hi/lo pairs, three tcgen05 MMAs into one fp32 accumulator; dense outputs within "
                      "1e-4 of the fp64 reference graph at 1024x1024 (tests/test_f16x3_gpu.py, measured 2.4e-5 R-50 / 2.8e-5 R-101)"
                      if precision == "f16x3" else "bf16 operands: ~1e-2 of max, NOT the parity arithmetic")
    if clocks is not None:
        line["clocks"] = clocks
    extras = not getattr(args, "no_extras", False)
    if extras and precision == "f16x3" and depth == 50:
        # the same configuration in single-pass bf16 arithmetic (3x the tensor rate, ~1e-2 accuracy), with the measured
        # detection-level difference against the parity arithmetic
        b16, det16, _ = run_config("r50", "bf16", batch, args, rank, world, local, benchmod, flush)
        b16["detection_diff_vs_f16x3"] = detection_diff(det16, det, img)
        line["bf16"] = b16
        del det16
        torch.cuda.empty_cache()
        # the reference's init_weights zeroes every bottleneck's last norm scale (zero_init_residual): the same configuration
        # with randomised norm scales instead (the weights of the 1024x1024 parity test), so that the headline is shown not
        # to depend on all-zero conv3 operands
        nz, detnz, _ = run_config("r50", precision, batch, args, rank, world, local, benchmod, flush, reference_init=False)
        nz["weights"] = "random_state_dict(50, reference_init=False): no zero_init_residual, norm scales U(0.5, 1.5)"
        line["nonzero_init"] = nz
        del detnz
        torch.cuda.empty_cache()
    if extras and depth == 50:
        # BASELINE.json configs[3] and [4]: R-101 at 4 tiles/GPU (batch 32 over 8 GPUs), Swin-T + DCN head at 8 tiles/GPU
        # (batch 64 over 8 GPUs) - both in the benchmarked arithmetic; Swin-T also in single-pass bf16 for reference
        cfgs = {}
        try:
            cfgs["r101_b4_per_gpu"], d2, _ = run_config("r101", precision, 4, args, rank, world, local, benchmod, flush)
            del d2
            torch.cuda.empty_cache()
            cfgs["swin_tiny_b8_per_gpu"], d3, _ = run_config("swin_tiny", precision, 8, args, rank, world, local, benchmod, flush)
            del d3
            torch.cuda.empty_cache()
            if precision != "bf16":
                cfgs["swin_tiny_b8_per_gpu_bf16"], d4, _ = run_config("swin_tiny", "bf16", 8, args, rank, world, local, benchmod, flush,
                                                                      steps=3)
                del d4
                torch.cuda.empty_cache()
        except Exception as ex:                                   # never lose the headline line to an extra
            cfgs["error"] = repr(ex)
        line["configs"] = cfgs
    return line
