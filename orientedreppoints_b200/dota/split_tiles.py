"""Tile producer: mirror of DOTA_devkit/SplitOnlyImage_multi_process.py (splitbase.SplitSingle :51-87,
saveimagepatches :38-49; the demo splits with gap=200, subsize=1024, rates 1 / 0.5 / 1.5 :113-118).

The reference writes every tile to `<name>__<rate>__<left>___<up>.png` and the test data loader decodes it again;
here the decoded image goes to the device once and the uint8 HWC tile batch the detector consumes is cut out in HBM by
one kernel (`orp_split_tiles_u8`).  Tile names and origins are the reference's, so `dota/result_merge.py` (which parses
`__<rate>__<left>___<up>`) maps the detections back unchanged.

`split_image(img, name, rate)` resizes on the host with the reference's own cv2.resize call.  `iter_tiles_multiscale`
is the multi-scale producer on the device: the original image is uploaded once and every tile of every rate is computed
from it by OpenCV's fixed-point bicubic arithmetic (`orp_resize_tiles_cubic_u8`, DESIGN.md §2 deviation 7).
"""
import ctypes

import numpy as np
import torch

from .. import _lib


def tile_origins(width, height, subsize=1024, gap=200):
    """(left, up) of every tile in the reference's order (left outer loop, up inner loop; the last tile of a row /
    column is pulled back so that it ends at the image border; SplitOnlyImage_multi_process.py:67-87)"""
    if subsize <= gap:
        raise ValueError("gap must be smaller than subsize")
    slide = subsize - gap
    out = []
    left = 0
    while left < width:
        if left + subsize >= width:
            left = max(width - subsize, 0)
        up = 0
        while up < height:
            if up + subsize >= height:
                up = max(height - subsize, 0)
            out.append((left, up))
            if up + subsize >= height:
                break
            up += slide
        if left + subsize >= width:
            break
        left += slide
    return out


def tile_names(name, rate, origins):
    """`<name>__<rate>__<left>___<up>` (SplitOnlyImage_multi_process.py:60,77; str(rate) as python prints it)"""
    base = name + '__' + str(rate) + '__'
    return [base + str(l) + '___' + str(u) for l, u in origins]


def resize_image(img, rate):
    """rate != 1: cv2.resize(..., fx=rate, fy=rate, interpolation=cv2.INTER_CUBIC) on the host, exactly the reference's
    call (:54-58) - a one-off per image, not on the per-tile path"""
    if rate == 1:
        return img
    import cv2
    return cv2.resize(np.asarray(img), None, fx=rate, fy=rate, interpolation=cv2.INTER_CUBIC)


def split_image(img, name="img", rate=1, subsize=1024, gap=200, device=None):
    """img: decoded uint8 HWC image (numpy array or tensor, host or device) -> (tiles uint8 [T,subsize,subsize,C] on the
    device, names, origins).  Windows leaving the image are zero padded (padding=True, :44-47)."""
    if not torch.is_tensor(img):
        img = torch.from_numpy(np.ascontiguousarray(resize_image(img, rate)))
    elif rate != 1:
        img = torch.from_numpy(np.ascontiguousarray(resize_image(img.cpu().numpy(), rate)))
    if img.dtype != torch.uint8 or img.dim() != 3:
        raise TypeError("split_image: uint8 HWC image expected")
    dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    img = img.to(dev).contiguous()
    h, w, c = img.shape
    origins = tile_origins(w, h, subsize, gap)
    org = torch.tensor(origins, dtype=torch.int32).reshape(-1, 2).to(dev)
    out = torch.empty((len(origins), subsize, subsize, c), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().orp_split_tiles_u8(_lib.ptr(img), h, w, c, _lib.ptr(org), len(origins), subsize, _lib.ptr(out),
                                                 _lib.current_stream_ptr()), "orp_split_tiles_u8")
    return out, tile_names(name, rate, origins), origins


# ---- multi-scale on the device: OpenCV's portable fixed-point INTER_CUBIC (DESIGN.md §2 deviation 7) ----

def scaled_size(width, height, rate):
    """(Wr, Hr) of cv2.resize(fx=fy=rate): saturate_cast<int>(n * rate), i.e. round half to even; empty is an error"""
    if not rate > 0:
        raise ValueError("rate must be > 0, got %r" % (rate,))
    wr, hr = round(width * float(rate)), round(height * float(rate))
    if wr < 1 or hr < 1:
        raise ValueError("%dx%d at rate %r resizes to an empty image" % (width, height, rate))
    return wr, hr


def _device(device):
    return torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)


def _check_image(img):
    if img.dtype != torch.uint8 or img.dim() != 3 or not 1 <= img.shape[2] <= 4:
        raise TypeError("uint8 HWC image with 1..4 channels expected")


def resize_tables(w, h, rates, device=None):
    """device coefficient tables of every rate != 1, concatenated in rate order (the layout
    orp_resize_tiles_cubic_u8 takes): (xidx int32 [sum Wr, 4], xw int16 [sum Wr, 4], yidx, yw)"""
    dev = _device(device)
    sizes = [scaled_size(w, h, r) for r in rates]
    nx = sum(s[0] for s, r in zip(sizes, rates) if r != 1)
    ny = sum(s[1] for s, r in zip(sizes, rates) if r != 1)
    xidx = torch.empty((nx, 4), dtype=torch.int32, device=dev)
    xw = torch.empty((nx, 4), dtype=torch.int16, device=dev)
    yidx = torch.empty((ny, 4), dtype=torch.int32, device=dev)
    yw = torch.empty((ny, 4), dtype=torch.int16, device=dev)
    ox = oy = 0
    with torch.cuda.device(dev):
        st = _lib.current_stream_ptr()
        for (wr, hr), r in zip(sizes, rates):
            if r == 1:
                continue
            _lib.check(_lib.lib().orp_resize_cubic_table(w, float(r), wr, _lib.ptr(xidx[ox:]), _lib.ptr(xw[ox:]), st),
                       "orp_resize_cubic_table")
            _lib.check(_lib.lib().orp_resize_cubic_table(h, float(r), hr, _lib.ptr(yidx[oy:]), _lib.ptr(yw[oy:]), st),
                       "orp_resize_cubic_table")
            ox, oy = ox + wr, oy + hr
    return xidx, xw, yidx, yw


def resize_image_device(img, rate):
    """device uint8 HWC tensor -> the image resized by `rate` on the device, cv2.resize(img, None, fx=rate, fy=rate,
    interpolation=INTER_CUBIC) under the fixed-point contract (within 1 LSB of cv2).  Rate 1 returns `img` itself."""
    if not torch.is_tensor(img) or not img.is_cuda:
        raise TypeError("resize_image_device: device tensor expected")
    _check_image(img)
    h, w, c = img.shape
    wr, hr = scaled_size(w, h, rate)
    if rate == 1:
        return img
    img = img.contiguous()
    xidx, xw, yidx, yw = resize_tables(w, h, [rate], img.device)
    out = torch.empty((hr, wr, c), dtype=torch.uint8, device=img.device)
    with torch.cuda.device(img.device):
        _lib.check(_lib.lib().orp_resize_cubic_u8(_lib.ptr(img), h, w, c, float(rate), _lib.ptr(xidx), _lib.ptr(xw),
                                                  _lib.ptr(yidx), _lib.ptr(yw), _lib.ptr(out), _lib.current_stream_ptr()),
                   "orp_resize_cubic_u8")
    return out


def iter_tiles_multiscale(img, name="img", rates=(0.5, 1.0, 1.5), subsize=1024, gap=200, batch=16, device=None):
    """Streaming multi-scale tile producer: yields (tiles uint8 [n <= batch, subsize, subsize, C] on the device, names,
    origins) in the reference's order - rates in the given order, each rate's tiles in `tile_origins` order, names
    `<name>__<str(rate)>__<left>___<up>` - with batches that run across rates.

    The original image goes to the device once (asynchronously from pinned memory when it comes from the host); every
    tile pixel is computed from it on the current stream, so the resized images are never materialised.  Device memory
    is the image, the tables and two batch buffers used in turn: a yielded batch is overwritten two batches later, so
    clone it to keep it."""
    rates = list(rates)
    if not 1 <= len(rates) <= _lib.ORP_RESIZE_MAX_RATES:
        raise ValueError("1 to %d rates expected" % _lib.ORP_RESIZE_MAX_RATES)
    if batch < 1:
        raise ValueError("batch must be >= 1")
    src = img if torch.is_tensor(img) else torch.from_numpy(np.ascontiguousarray(img))
    _check_image(src)
    h, w, c = src.shape
    per_rate = []
    for r in rates:
        wr, hr = scaled_size(w, h, r)
        org = tile_origins(wr, hr, subsize, gap)
        per_rate.append((r, org, tile_names(name, r, org)))
    dev = _device(device)
    with torch.cuda.device(dev):
        if src.device.type == 'cpu':
            src = src.contiguous().pin_memory().to(dev, non_blocking=True)
        else:
            src = src.to(dev).contiguous()
        xidx, xw, yidx, yw = resize_tables(w, h, rates, dev)
        desc = [(i, l, u) for i, (_, org, _) in enumerate(per_rate) for (l, u) in org]
        desc_dev = torch.tensor(desc, dtype=torch.int32).reshape(-1, 3).pin_memory().to(dev, non_blocking=True)
        bufs = [torch.empty((min(batch, len(desc)), subsize, subsize, c), dtype=torch.uint8, device=dev)
                for _ in range(min(2, -(-len(desc) // batch)))]
    names = [n for _, _, nm in per_rate for n in nm]
    origins = [o for _, org, _ in per_rate for o in org]
    rates_c = (ctypes.c_double * len(rates))(*[float(r) for r in rates])
    for k, i in enumerate(range(0, len(desc), batch)):
        n = min(batch, len(desc) - i)
        out = bufs[k % len(bufs)][:n]
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().orp_resize_tiles_cubic_u8(
                _lib.ptr(src), h, w, c, len(rates), rates_c, _lib.ptr(xidx), _lib.ptr(xw), _lib.ptr(yidx), _lib.ptr(yw),
                _lib.ptr(desc_dev[i:]), n, subsize, _lib.ptr(out), _lib.current_stream_ptr()), "orp_resize_tiles_cubic_u8")
        yield out, names[i:i + n], origins[i:i + n]
