"""Inputs of the denoiser computed from the photo on the GPU.

``photo_to_y512(photo)``: the 512x512 conditioning image ``y512`` that the reference loader builds on the host as
``cv2.resize(rgb_u8, (512, 512), INTER_LINEAR) / 255`` (datasets/doc_dataset/doc_benchmark.py:68-81), byte for byte, in one launch
for a uint8 NHWC batch or a list of photos of different sizes.
"""
from __future__ import annotations

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
