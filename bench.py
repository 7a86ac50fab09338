#!/usr/bin/env python
"""bench.py - measurement harness of the OrientedRepPoints B200 hot path (contract in the task brief).

    python bench.py --gpus 1 --steps 20 --warmup 5                 # our arm, one JSON line
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1 # reference CPU arm, one JSON line
    torchrun ... bench.py --gpus N ...                             # one rank per GPU (weak scaling)

A "step" is one pass of the hot path over one batch of synthetic input:
  workload r50_tile (default once the dense path is built): one 1024x1024 tile through R-50 + FPN +
      OrientedRepPointsHead + minaerarect + multiclass_rnms (BASELINE.json configs[1]); metric tiles/s.
  workload nms_100k: rotated NMS (thr 0.1) over 100k synthetic proposals in a 1024^2 extent
      (BASELINE.json configs[2] at its 100k point); metric Mpairs/s with pairs = N(N-1)/2.
Timing: CUDA events on the launching stream around every step, an L2 flush (write of a 512 MiB buffer)
between timed steps, barrier + synchronize on both sides of the timed region, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, help="r50_tile | nms_100k | nms_100k_sparse")
    ap.add_argument("--boxes", type=int, default=100000)
    ap.add_argument("--batch", type=int, default=None, help="tiles per step per GPU (r50_tile)")
    ap.add_argument("--precision", default=None, help="r50_tile arithmetic: f16x3 (default: tensor cores, fp32-faithful) | bf16 | fp32")
    ap.add_argument("--no-extras", dest="no_extras", action="store_true",
                    help="r50_tile: skip the extra objects of the line (bf16 arithmetic, R-101 / Swin-T configs, NMS sweep)")
    ap.add_argument("--backbone", default=None, help="r50_tile workload backbone: r50 (default) | r101 | swin_tiny")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", dest="no_graph", action="store_true", help="r50_tile: eager launches instead of a CUDA graph")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 or "
                         "float64, at most 64 MiB in all); the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT = 64 << 20                                              # bytes --dump-outputs writes at most


def write_outputs(path, arrays):
    """--dump-outputs: every array as path/<name>.npy, float32 as it is and anything else as float64"""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: (a if a.dtype == np.float32 else a.astype(np.float64)) for k, a in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- helpers
def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                    "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ----------------------------------------------------------------------------------------------- NMS workload
def nms_bitmatrix_bytes(n):
    """SURVEY.md 8(d): bytes of the REFERENCE's formulation (boxes 36 N + 64-bit mask write and read 16 N ceil(N/64),
    ~0.5 B per pair).  This kernel never materialises that matrix; the figure is reported for context only."""
    return 36.0 * n + 16.0 * n * ((n + 63) // 64)


# per-candidate-pair arithmetic of the exact decision (fp32 Sutherland-Hodgman of two quadrilaterals in pair-local
# coordinates with a running error bound: 4 clip edges x <=8 ring vertices x ~14 flops + areas), counted from the source
CLIP_FLOPS = 700.0
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 x 1.965 GHz = 74.4 (nominal, no measured figure)


def time_nms(dets_h, local, steps, warm, world, flush, thr=0.1):
    """device-timed rotated NMS of one box set resident in HBM: (ms per call, sweep-kernel ms, kept, stats, kept indices of
    the last call)"""
    import torch
    from orientedreppoints_b200 import _lib
    from orientedreppoints_b200.ops import rnms_indices
    dev = torch.device("cuda", local)
    dets = torch.from_numpy(dets_h).to(dev)
    _lib.set_timing(True)
    for _ in range(warm):
        rnms_indices(dets, thr, order=_lib.ORP_ORDER_SCORE_DESC, return_count_tensor=True)
    barrier(world)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sweep = []
    for s in range(steps):
        flush.fill_(s & 0xFF)                                              # L2 flush, not timed
        ev[s][0].record()
        keep, cnt = rnms_indices(dets, thr, order=_lib.ORP_ORDER_SCORE_DESC, return_count_tensor=True)
        ev[s][1].record()
        torch.cuda.current_stream().synchronize()
        sweep.append(_lib.last_sweep_ms())
    _lib.set_timing(False)
    ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) / steps, world)
    kept = int(cnt.item())
    return ms, float(np.mean(sweep)), kept, _lib.last_nms_stats(), keep[:kept].cpu().numpy()


def nms_sweep(args, rank, world, local, sizes=(10000, 20000, 50000, 100000, 200000)):
    """BASELINE.json configs[2]: poly_nms over 10k -> 200k rotated proposals, IoU thr 0.1, at constant density (1k boxes
    per 1024^2) and dense (everything inside one 1024^2 extent); every rank processes its own sets (weak scaling)."""
    import torch
    from orientedreppoints_b200 import _lib
    from orientedreppoints_b200.dota.poly_nms_gpu import poly_gpu_nms
    from orientedreppoints_b200.synth import const_density_extent, gen_rotated_boxes
    dev = torch.device("cuda", local)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    pk = peaks()
    rows = []
    head = None
    for n in sizes:
        for dense in (False, True):
            d = gen_rotated_boxes(n, seed=100 + rank, extent=1024.0 if dense else const_density_extent(n))
            ms, sweep_ms, kept, st, _ = time_nms(d, local, 5, 3, world, flush)
            pairs = n * (n - 1) / 2.0
            row = {"n": n, "variant": "dense_1024" if dense else "const_density", "ms": ms, "Mpairs_per_s": world * pairs / (ms * 1e-3) / 1e6,
                   "kept": kept, "sweep_kernel_ms": sweep_ms, "pairs_swept": st["pairs_total"], "pairs_aabb": st["pairs_aabb"],
                   "candidates": st["edges"], "pairs_clipped": st["pairs_clipped"], "pairs_fp64": st["pairs_fp64"],
                   "suppressing": st["suppressing"], "rounds": st["rounds"], "overflow": st["overflow"],
                   "prefilter_hit_rate": st["pairs_aabb"] / pairs,
                   "clip_tflops": st["pairs_clipped"] * CLIP_FLOPS / (ms * 1e-3) / 1e12}
            rows.append(row)
            if n == 100000 and dense:
                head = (d, row)
    out = {"workload": "poly_nms sweep, IoU thr 0.1, one set per GPU per call, L2 flushed between calls, device timed (CUDA events)",
           "unit": "Mpairs/s (pairs = N(N-1)/2)", "n_gpus": world, "sweep": rows}
    if head is not None:
        d, row = head
        for _ in range(2):
            poly_gpu_nms(d, 0.1, device_id=local)
        barrier(world)
        t0 = time.perf_counter()
        reps = 5
        for _ in range(reps):
            kl = poly_gpu_nms(d, 0.1, device_id=local)
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / reps, world)
        pairs = 100000 * 99999 / 2.0
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_nms_traffic_dense100k.json")))
            traffic = tj                                                  # ncu dram bytes of the kernels of one call
        except Exception:
            pass
        out["headline_100k_dense"] = {
            "value": row["Mpairs_per_s"], "unit": "Mpairs/s", "ms": row["ms"], "kept": row["kept"],
            "e2e": {"value": world * pairs / (e2e_ms * 1e-3) / 1e6, "unit": "Mpairs/s", "ms": e2e_ms,
                    "h2d_bytes_per_step": int(d.nbytes), "d2h_bytes_per_step": int(len(kl) * 8 + 4),
                    "api": "DOTA_devkit.poly_nms_gpu.poly_gpu_nms(np.float32[N,9], thr) -> list"},
            "roofs": {
                "note": "the reference formulation (N x N/64 bit matrix, %.2f GB at 100k) is never materialised: candidate pairs "
                        "come from an x-sweep with exact-safe bounds and only (undecided box, kept candidate) pairs are clipped, "
                        "so neither HBM nor the fp32 pipe is close to its roof - the call is bound by sort / scan / grid-sync "
                        "latency and by the divergent clip" % (nms_bitmatrix_bytes(100000) / 1e9),
                "reference_formulation_bytes": nms_bitmatrix_bytes(100000),
                "reference_formulation_GBps_equiv": nms_bitmatrix_bytes(100000) / (row["ms"] * 1e-3) / 1e9,
                "hbm_peak_GBps": pk["hbm_gbs"], "dram_traffic_ncu": traffic,
                "clip_tflops": row["clip_tflops"], "fp32_peak_tflops_nominal": FP32_PEAK_TFLOPS,
                "clip_frac_of_fp32_peak": row["clip_tflops"] / FP32_PEAK_TFLOPS}}
    return out


def run_nms(args, rank, world, local, dense=True):
    """--workload nms_100k / nms_100k_sparse: the NMS half of the BASELINE metric as its own JSON line"""
    import torch
    from orientedreppoints_b200 import _lib
    from orientedreppoints_b200.dota.poly_nms_gpu import poly_gpu_nms
    from orientedreppoints_b200.synth import const_density_extent, gen_rotated_boxes
    n = args.boxes
    dets_h = gen_rotated_boxes(n, seed=100 + rank, extent=1024.0 if dense else const_density_extent(n))   # per-rank set: weak scaling
    dev = torch.device("cuda", local)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    thr = 0.1
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.reset_launch_count()
    ms, sweep_avg, kept, stats, keep = time_nms(dets_h, local, args.steps, max(args.warmup, 3), world, flush, thr)
    launches = _lib.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"keep": keep})
    pairs = n * (n - 1) / 2.0
    for _ in range(2):
        poly_gpu_nms(dets_h, thr, device_id=local)
    barrier(world)
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(e2e_steps):
        kl = poly_gpu_nms(dets_h, thr, device_id=local)
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps, world)
    assert len(kl) == kept
    pk = peaks()
    clip_tf = stats["pairs_clipped"] * CLIP_FLOPS / (ms * 1e-3) / 1e12
    line = {
        "metric": "rotated IoU+NMS Mpairs/sec", "value": world * pairs / (ms * 1e-3) / 1e6,
        "unit": "Mpairs/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (+f64 inside the decision band)", "data": "synthetic",
        "config": {"workload": "poly_nms %d rotated proposals in %s, IoU thr 0.1, one set per GPU" %
                   (n, "a 1024x1024 extent (dense)" if dense else "constant 1k/1024^2 density"),
                   "l2": "512 MiB flush write between timed steps", "kept": kept,
                   "pairs_swept": stats["pairs_total"], "pairs_aabb": stats["pairs_aabb"], "candidates": stats["edges"],
                   "pairs_clipped": stats["pairs_clipped"], "pairs_fp64": stats["pairs_fp64"],
                   "suppressing": stats["suppressing"], "rounds": stats["rounds"], "overflow": stats["overflow"],
                   "prefilter_hit_rate": stats["pairs_aabb"] / pairs},
        "gpu_launches": int(launches),
        "e2e": {"value": world * pairs / (e2e_ms * 1e-3) / 1e6, "unit": "Mpairs/s",
                "h2d_bytes_per_step": int(dets_h.nbytes), "d2h_bytes_per_step": int(kept * 8 + 4),
                "api": "DOTA_devkit.poly_nms_gpu.poly_gpu_nms(np.float32[N,9], thr) -> list"},
        "roofline": {"bound": "hbm", "kernel": "nms_sweep_kernel", "achieved": None, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": None, "traffic": None, "peak_source": pk["source"],
                     "note": "HBM is not the binding roof of this formulation (no N^2 bit matrix): see clip_tflops and "
                             "reference_formulation_GBps_equiv; dram bytes of a call are in profiles/ (ncu)",
                     "reference_formulation_bytes": nms_bitmatrix_bytes(n),
                     "reference_formulation_GBps_equiv": nms_bitmatrix_bytes(n) / (ms * 1e-3) / 1e9,
                     "clip_tflops": clip_tf, "clip_frac_of_fp32_peak": clip_tf / FP32_PEAK_TFLOPS,
                     "kernel_ms": sweep_avg, "kernel_share_of_step": sweep_avg / ms},
    }
    if clocks is not None:
        line["clocks"] = clocks
    return line


# ----------------------------------------------------------------------------------------------- reference arm
def cpu_baseline_block(n_boxes, shards):
    from oracle import ref_driver
    b = ref_driver.timed_baseline(n_boxes, 0.1, shards)
    return {"value": b["value"], "unit": "Mpairs/s", "cores": b["cores"], "kind": b["kind"], "sample": b["sample"],
            "seconds": b["seconds"]}


def run_reference_tile(args, rank, world):
    """Tile workload on the host cores: the PyTorch fp32 re-declaration of the reference graph (the reference package
    itself cannot be imported here: mmcv 0.6.2 / timm / pycocotools are absent) + the restated reference
    post-processing over the CPU oracle (minaerarect, fp64 polyiou NMS with the reference's own AABB prefilter).
    kind = "port".  One 1024x1024 tile per step, every host thread torch can use."""
    if rank != 0:
        return None
    import torch
    from oracle import torch_reference as tr
    from orientedreppoints_b200.weights import random_state_dict
    avail = os.cpu_count() or 1
    # torch's CPU convolutions stop scaling (and regress) far below the 128 threads of the GPU box: measured 47 s per
    # tile with 128 threads against 7.8 s with 8; 32 threads is what a tuned CPU deployment of the reference would use
    cores = min(avail, 32)
    torch.set_num_threads(cores)
    sd = random_state_dict(50, seed=0, reference_init=True)
    tile_u8 = torch.randint(0, 256, (1, 1024, 1024, 3), generator=torch.Generator().manual_seed(1000), dtype=torch.uint8)
    mean = torch.tensor([123.675, 116.28, 103.53]); stdinv = 1.0 / torch.tensor([58.395, 57.12, 57.375])

    def step():
        with torch.no_grad():
            # Normalize (to_rgb, mean, std) + ImageToTensor of the test pipeline, as the reference does them on the host
            img = ((tile_u8.float().flip(-1) - mean) * stdinv).permute(0, 3, 1, 2).contiguous()
            outs, _ = tr.forward_dense(sd, img)
            return tr.get_bboxes_single([o[0][0] for o in outs], [o[2][0] for o in outs], score_thr=0.0)

    # a CPU step takes seconds to tens of seconds: keep the whole run within ~3 minutes (at most one warm-up step, then as
    # many of the requested timed steps as fit; the line reports how many were timed)
    budget = 180.0
    t_begin = time.perf_counter()
    if args.warmup > 0:
        step()
    ts = []
    for i in range(max(1, args.steps)):
        t0 = time.perf_counter()
        dets, _ = step()
        ts.append(time.perf_counter() - t0)
        if (time.perf_counter() - t_begin) + ts[-1] > budget:
            break
    sec = float(np.mean(ts))
    sample = ("1 synthetic 1024x1024 tile per step, R-50 FPN OrientedRepPoints fp32 on %d host threads (torch re-declaration of "
              "the reference graph + CPU oracle post-processing, score_thr=0), %d detections" % (cores, int(dets.shape[0])))
    return {"impl": "reference", "metric": "1024x1024 tiles/sec", "value": 1.0 / sec, "unit": "tiles/s", "n_gpus": args.gpus,
            "steps": len(ts), "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (+f64 geometry)", "data": "synthetic",
            "config": {"workload": "bounded sample of the tile workload: " + sample,
                       "steps_requested": args.steps, "warmup_requested": args.warmup, "time_budget_s": budget},
            "cpu_baseline": {"value": 1.0 / sec, "unit": "tiles/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": 1.0 / sec, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def run_reference(args, rank, world):
    """the reference's own CPU implementation of the geometry path on the host cores"""
    if rank != 0:
        return None
    cores = os.cpu_count() or 1
    shards = max(1, min(cores, 16))
    vals, secs = [], []
    nb = 1500
    for _ in range(args.warmup):
        cpu_baseline_block(300, shards)
    last = None
    for _ in range(args.steps):
        last = cpu_baseline_block(nb, shards)
        vals.append(last["value"])
        secs.append(last["seconds"])
    v = float(np.mean(vals))
    return {"impl": "reference", "metric": "rotated IoU+NMS Mpairs/sec", "value": v, "unit": "Mpairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "bounded sample of the poly_nms workload: " + last["sample"]},
            "cpu_baseline": {"value": v, "unit": "Mpairs/s", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": v, "unit": "Mpairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    args = parse_args()
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if (args.workload or "r50_tile") == "r50_tile":
            line = run_reference_tile(args, rank, world)
        else:
            line = run_reference(args, rank, world)
        if line is not None:
            print(json.dumps(line))
        return 0
    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "bench.py needs a GPU: the product path has no CPU fallback"}))
        return 1
    rank, world, local = dist_setup(args.gpus)
    workload = args.workload
    if workload is None:
        try:
            from orientedreppoints_b200 import bench_tile  # noqa: F401  (dense path present?)
            workload = "r50_tile"
        except ImportError:
            workload = "nms_100k"
    if workload == "r50_tile":
        from orientedreppoints_b200 import bench_tile
        line = bench_tile.run(args, rank, world, local, sys.modules[__name__])
        if not args.no_extras:
            # the second half of the BASELINE metric ("rotated IoU+NMS Mpairs/sec") rides on the same line
            try:
                line["nms"] = nms_sweep(args, rank, world, local)
            except Exception as ex:
                line["nms"] = {"error": repr(ex)}
    elif workload in ("nms_100k", "nms_100k_sparse"):
        line = run_nms(args, rank, world, local, dense=(workload == "nms_100k"))
    else:
        raise SystemExit("unknown workload " + workload)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        if workload == "r50_tile":
            class _A:
                pass
            a = _A()
            a.warmup, a.steps, a.gpus = 0, 1, 1
            ref = run_reference_tile(a, 0, 1)
            line["cpu_baseline"] = dict(ref["cpu_baseline"], seconds=ref["ms_per_step"] / 1e3)
            line["cpu_baseline_geometry"] = cpu_baseline_block(2000, 1)      # the reference's compiled polyiou under its NMS loop
        else:
            line["cpu_baseline"] = cpu_baseline_block(2000, 1)
        line["cpu_baseline"]["host_cores_available"] = cores
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
