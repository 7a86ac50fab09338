"""Whole-image inference: tile producer -> detector -> ResultMerge, device resident between the steps.

Composition of the three reference stages that bracket the hot path (SURVEY 8 rows n4, a1-a12, n1):
  DOTA_devkit/SplitOnlyImage_multi_process.py (tiles, gap 200)        -> dota/split_tiles.py
  tools/test.py + OrientedRepPointsDetector.simple_test per tile      -> detector.py
  tools/parse_pkl/parse_pkl_mege_results_for_dota_evaluation.py:93-192 (Task1 lines per class) +
  DOTA_devkit/ResultMerge_multi_process.py:182-262 (coordinates back to the image, per-image poly NMS thr 0.1)
                                                                      -> dota/result_merge.py
The reference goes through PNG tiles, a pickle and per-class text files between these stages; here the tiles never
leave HBM and the per-class result lines are merged in memory (the same `merge_lines` the file-based mirror uses).
"""
from .result_merge import merge_lines
from .split_tiles import iter_tiles_multiscale, split_image

# mmdet/datasets/dota.py:8-12
DOTA_CLASSES = ('plane', 'baseball-diamond', 'bridge', 'ground-track-field', 'small-vehicle', 'large-vehicle', 'ship',
                'tennis-court', 'basketball-court', 'storage-tank', 'soccer-ball-field', 'roundabout', 'harbor',
                'swimming-pool', 'helicopter')


def task1_lines(results, tile_names):
    """rbbox2result lists of every tile -> per-class lists of `tilename score x1 y1 ... x4 y4` (the lines
    parse_pkl_mege_results_for_dota_evaluation.py:150-187 writes: bbox[-1] is the score, bbox[-9:-1] the quadrilateral)"""
    per_class = [[] for _ in DOTA_CLASSES]
    for res, tname in zip(results, tile_names):
        for c, arr in enumerate(res):
            for bbox in arr:
                per_class[c].append(tname + ' ' + str(float(bbox[-1])) + ' ' + ' '.join(str(float(v)) for v in bbox[-9:-1]))
    return per_class


def detect_image(det, img_u8, name="P0000", rate=1, subsize=1024, gap=200, batch=16, merge_thresh=None):
    """det: OrientedRepPointsDetector; img_u8: decoded uint8 HWC image (numpy or tensor).  Returns
    {class name: [`imgname score x1 y1 x2 y2 x3 y3 x4 y4`, ...]} in the Task1 format after ResultMerge."""
    tiles, names, _ = split_image(img_u8, name, rate, subsize, gap, device=det.device)
    results = []
    for i in range(0, tiles.shape[0], batch):
        results.extend(det.simple_test(tiles[i:i + batch]))
    per_class = task1_lines(results, names)
    return {cname: merge_lines(lines, merge_thresh) for cname, lines in zip(DOTA_CLASSES, per_class)}


def detect_image_multiscale(det, img_u8, name="P0000", rates=(0.5, 1.0, 1.5), subsize=1024, gap=200, batch=16,
                            merge_thresh=None):
    """The reference's multi-scale test of one image: tiles of every rate (SplitOnlyImage_multi_process.py splitdata(rate)
    per rate, here one streaming device producer over the original image) -> detector -> ONE ResultMerge over the tiles
    of all rates (mergebypoly over the parsed pickle; poly2origpoly divides by each tile's rate).  Returns
    {class name: [`imgname score x1 y1 x2 y2 x3 y3 x4 y4`, ...]} like detect_image."""
    results, names = [], []
    for tiles, tnames, _ in iter_tiles_multiscale(img_u8, name, rates, subsize, gap, batch, device=det.device):
        results.extend(det.simple_test(tiles))
        names.extend(tnames)
    per_class = task1_lines(results, names)
    return {cname: merge_lines(lines, merge_thresh) for cname, lines in zip(DOTA_CLASSES, per_class)}
