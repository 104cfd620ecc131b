"""Inputs decoded and computed on the GPU.

``decode_jpeg(files, device)``: JPEG files to uint8 HWC RGB photos on the GPU, byte-equal to
``cv2.imdecode(buf, cv2.IMREAD_COLOR)[..., ::-1]`` (the reference loader's ``cv2.imread`` -> RGB, EXIF orientation applied), one
upload and one planned decode for a batch of any sizes.

``photo_to_y512(photo)``: the 512x512 conditioning image ``y512`` that the reference loader builds on the host as
``cv2.resize(rgb_u8, (512, 512), INTER_LINEAR) / 255`` (datasets/doc_dataset/doc_benchmark.py:68-81), byte for byte, in one launch
for a uint8 NHWC batch or a list of photos of different sizes.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def table_bytes(max_docs: int) -> int:
    """bytes of a y512 table for up to `max_docs` documents"""
    return _lib.lib().dvd_y512_table_bytes(max_docs)


def plan_y512(table_host: torch.Tensor, photos) -> None:
    """Plans the y512 launch of uint8 HWC device photos [H,W,3] (document i: photos[i]) into the host tensor `table_host` (uint8,
    pinned for an async upload, at least ``table_bytes(len(photos))`` bytes).  No CUDA call."""
    n = len(photos)
    docs = (_lib.Y512Doc * max(n, 1))(*[_lib.Y512Doc(p.data_ptr(), p.shape[0], p.shape[1]) for p in photos])
    _lib.check(_lib.lib().dvd_y512_u8_plan(docs if n else None, n, _lib.ptr(table_host), table_host.numel()), "dvd_y512_u8_plan")


def launch_y512(table: torch.Tensor, y512: torch.Tensor) -> None:
    """one launch on the current stream: documents 0..n-1 of y512 [>= n,3,512,512] fp32 from the uploaded plan `table`"""
    _lib.check(_lib.lib().dvd_y512_u8(_lib.ptr(table), _lib.ptr(y512), _lib.stream_ptr()), "dvd_y512_u8")


def check_photos(photos, device: torch.device | None = None) -> list:
    """list of uint8 HWC RGB photos (contiguous, at least 1x1, on one CUDA device) or a ValueError / RuntimeError"""
    photos = list(photos)
    for i, p in enumerate(photos):
        if not isinstance(p, torch.Tensor) or p.dtype != torch.uint8 or p.dim() != 3 or p.shape[2] != 3 or p.shape[0] < 1 or p.shape[1] < 1:
            raise ValueError(f"photo {i}: expected a uint8 HWC tensor with 3 channels, got "
                             f"{getattr(p, 'dtype', type(p))} {tuple(getattr(p, 'shape', ()))}")
        if not p.is_cuda:
            raise RuntimeError(f"photo {i} is on {p.device}: photo_to_y512 runs on the GPU only (dvd_b200 has no CPU path)")
        if not p.is_contiguous():
            raise ValueError(f"photo {i} is not contiguous")
        if p.device != (device or photos[0].device):
            raise ValueError(f"photo {i} is on {p.device}, photo 0 on {photos[0].device}")
    return photos


@torch.no_grad()
def photo_to_y512(photo, out: torch.Tensor | None = None) -> torch.Tensor:
    """The denoiser's y512 [B,3,512,512] fp32 from uint8 RGB photos, equal to
    ``torch.from_numpy(cv2.resize(photo_i, (512, 512), interpolation=cv2.INTER_LINEAR)).permute(2, 0, 1).float() / 255``.

    ``photo`` is a uint8 NHWC device tensor [B,H,W,3] or a list of B uint8 HWC device tensors [H_i,W_i,3] of any sizes; either
    way the result comes from one launch.  ``out`` (fp32 [B,3,512,512], contiguous, on the photos' device) receives it if given."""
    if isinstance(photo, (list, tuple)):
        photos = check_photos(photo)
    elif isinstance(photo, torch.Tensor):
        if photo.dtype != torch.uint8 or photo.dim() != 4 or photo.shape[3] != 3:
            raise ValueError(f"photo_to_y512 takes uint8 NHWC [B,H,W,3] or a list of uint8 HWC photos, got {photo.dtype} "
                             f"{tuple(photo.shape)}")
        photos = check_photos(photo.contiguous().unbind(0))
    else:
        raise ValueError(f"photo_to_y512 takes a uint8 tensor or a list of them, got {type(photo).__name__}")
    if not photos:
        raise ValueError("photo_to_y512: no photos")
    dev = photos[0].device
    shape = (len(photos), 3, 512, 512)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    elif out.dtype != torch.float32 or tuple(out.shape) != shape or not out.is_contiguous() or out.device != dev:
        raise ValueError(f"out must be a contiguous float32 tensor {shape} on {dev}, got {out.dtype} {tuple(out.shape)} on {out.device}")
    with torch.cuda.device(dev):
        table = _lib.PlannedTable(table_bytes(len(photos)), dev).upload(lambda host: plan_y512(host, photos))
        launch_y512(table, out)
    return out


# ---- JPEG decode ----
def jpeg_table_bytes(max_docs: int) -> int:
    """bytes of a JPEG decode table for up to `max_docs` files"""
    return _lib.lib().dvd_jpeg_table_bytes(max_docs)


def jpeg_workspace_bytes(max_docs: int, max_pixels: int, max_jpeg_bytes: int) -> int:
    """decode workspace for up to `max_docs` files with at most `max_pixels` pixels and `max_jpeg_bytes` bytes in all (each with
    sides within about 1:5)"""
    return _lib.lib().dvd_jpeg_workspace_bytes(max_docs, max_pixels, max_jpeg_bytes)


def _jpeg_docs(files, arena=None, offsets=None, outs=None):
    n = len(files)
    views = [memoryview(f).cast("B") for f in files]
    keep = [(C.c_uint8 * len(v)).from_buffer_copy(v) if v.readonly else (C.c_uint8 * len(v)).from_buffer(v) for v in views]
    docs = (_lib.JpegDoc * max(n, 1))()
    for i, k in enumerate(keep):
        docs[i].file_host = C.addressof(k) if len(k) else None
        docs[i].bytes = len(k)
        if arena is not None:
            docs[i].file = arena.data_ptr() + offsets[i]
            docs[i].out = outs[i].data_ptr()
    return docs, keep


def plan_jpeg(files, table_host: torch.Tensor | None = None, workspace_bytes: int = 0, arena: torch.Tensor | None = None,
              offsets=None, outs=None) -> list:
    """Parses the JPEG `files` (bytes-like) and returns the (H, W) of each decoded photo, after its EXIF orientation.  With
    `table_host` it also plans the decode of file i, stored in the device `arena` at offsets[i], into outs[i] (uint8 [H,W,3]).  No
    CUDA call.  A file the decoder does not take raises ValueError with the reason."""
    n = len(files)
    docs, keep = _jpeg_docs(files, arena, offsets, outs)
    hw = (C.c_int32 * max(2 * n, 1))()
    rc = _lib.lib().dvd_jpeg_plan(docs if n else None, n, _lib.ptr(table_host), 0 if table_host is None else table_host.numel(),
                                  workspace_bytes, hw)
    if rc != 0:
        raise ValueError(_lib.lib().dvd_last_error().decode(errors="replace"))
    del keep
    return [(hw[2 * i], hw[2 * i + 1]) for i in range(n)]


def jpeg_hw(files) -> list:
    """(H, W) of each JPEG file after its EXIF orientation, as decode_jpeg returns it (ValueError for a file it does not take)"""
    return plan_jpeg(list(files))


def pack_jpeg(files, host: torch.Tensor) -> list:
    """copies the files into the uint8 tensor `host` at 16-byte aligned offsets; returns the offsets"""
    offsets, off = [], 0
    for f in files:
        n = memoryview(f).nbytes
        if off + n > host.numel():
            raise ValueError(f"the files need more than the {host.numel()} bytes of the staging block")
        host[off:off + n] = torch.frombuffer(bytearray(f) if memoryview(f).readonly else f, dtype=torch.uint8)
        offsets.append(off)
        off = (off + n + 15) & ~15
    return offsets


def launch_jpeg(table: torch.Tensor, workspace: torch.Tensor) -> None:
    """the decode of the uploaded plan `table` on the current stream"""
    _lib.check(_lib.lib().dvd_jpeg_decode(_lib.ptr(table), _lib.ptr(workspace), _lib.stream_ptr()), "dvd_jpeg_decode")


@torch.no_grad()
def decode_jpeg(files, device, out=None) -> list:
    """JPEG files (bytes-like) -> list of uint8 HWC RGB tensors on `device`, photo i equal to
    ``cv2.imdecode(np.frombuffer(files[i], np.uint8), cv2.IMREAD_COLOR)[..., ::-1]``.

    Baseline and extended sequential 8-bit Huffman files with one interleaved scan (YCbCr 4:4:4, 4:2:2, 4:2:0 or grayscale, with or
    without restart intervals) are decoded; any other file raises ValueError naming the reason, and is for the caller to decode on
    the host.  The files are packed into one pinned block, copied with one async copy and decoded by one planned launch sequence on
    the current stream.  ``out`` (a list of contiguous uint8 [H,W,3] tensors on `device`, see ``jpeg_hw``) receives the photos if
    given."""
    files = list(files)
    if not files:
        raise ValueError("decode_jpeg: no files")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"decode_jpeg decodes on a CUDA device, got {dev} (dvd_b200 has no CPU path)")
    hw = jpeg_hw(files)
    with torch.cuda.device(dev):
        if out is None:
            out = [torch.empty((H, W, 3), dtype=torch.uint8, device=dev) for H, W in hw]
        else:
            out = list(out)
            if len(out) != len(files):
                raise ValueError(f"out has {len(out)} tensors for {len(files)} files")
            for i, (o, (H, W)) in enumerate(zip(out, hw)):
                if (not isinstance(o, torch.Tensor) or o.dtype != torch.uint8 or tuple(o.shape) != (H, W, 3) or not o.is_contiguous()
                        or o.device != dev):
                    raise ValueError(f"out[{i}] must be a contiguous uint8 tensor {(H, W, 3)} on {dev}")
        total = sum((memoryview(f).nbytes + 15) & ~15 for f in files)
        host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        offsets = pack_jpeg(files, host)
        arena = host.to(dev, non_blocking=True)
        # the padded sizes as the pixel bound hold for any aspect ratio
        ws_bytes = jpeg_workspace_bytes(len(files), sum((H + 15) * (W + 15) for H, W in hw), total)
        workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        table = _lib.PlannedTable(jpeg_table_bytes(len(files)), dev).upload(
            lambda t: plan_jpeg(files, t, ws_bytes, arena, offsets, out))
        launch_jpeg(table, workspace)
    return out
