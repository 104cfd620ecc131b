"""Unwarp operators with the reference's call surface.

* ``register_model2`` / ``SpatialTransformer2``  (datasets/utils/warping.py:14-73): generic bilinear
  ``grid_sample`` (align_corners=True, zeros padding) — ``reg_model_bilin([img, grid]) -> img``.
* ``dewarp_fullres(map64, photo)``: evaluation.py:300-306 + visualization_utils.py:75-77 fused into
  ONE bandwidth-bound kernel (no materialised full-resolution grid).  ``photo`` may also be a list of uint8 HWC photos of
  different sizes: they are dewarped in one launch.  ``size=(Ho, Wo)`` writes uint8 pages at a requested size instead of the
  photo's, supersampled when shrinking (the reference chain at ``s*Ho x s*Wo``, averaged over s x s blocks).
"""
from __future__ import annotations

from ctypes import byref, c_int32 as C_int32, c_longlong as C_longlong

import torch
import torch.nn as nn

from . import _lib

AFFINE = 0.987          # evaluation.py:306


def _chk(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: dvd_b200 has no CPU path")


class SpatialTransformer2(nn.Module):
    def __init__(self, size=None, mode="bilinear"):
        super().__init__()
        if mode != "bilinear":
            raise NotImplementedError("only bilinear sampling is on the val_TDiff path")
        self.mode = mode

    @torch.no_grad()
    def forward(self, src, flow):
        _chk(src, "src"); _chk(flow, "flow")
        src = src.float().contiguous(); flow = flow.float().contiguous()
        B, Cc, H, W = src.shape
        Bo, two, Ho, Wo = flow.shape
        assert two == 2 and Bo == B
        out = torch.empty((B, Cc, Ho, Wo), dtype=torch.float32, device=src.device)
        with torch.cuda.device(src.device):
            _lib.check(_lib.lib().dvd_grid_sample_f32(_lib.ptr(src), _lib.ptr(flow), _lib.ptr(out), B, Cc, H, W, Ho, Wo,
                                                      _lib.stream_ptr()), "dvd_grid_sample_f32")
        return out


class register_model2(nn.Module):                    # noqa: N801 (reference name)
    def __init__(self, img_size=(64, 1024, 1024), mode="bilinear"):
        super().__init__()
        self.spatial_trans = SpatialTransformer2(img_size, mode)

    def forward(self, x):
        return self.spatial_trans(x[0], x[1])


def plan_mixed(table_host: torch.Tensor, photos, outs, mh: int, mw: int, affine: float = AFFINE, C: int = 3) -> int:
    """Plans a mixed-size uint8 HWC batch (document i: photos[i] -> outs[i], device tensors [H,W,C]) into the host tensor
    `table_host` (pinned uint8, at least ``table_bytes(len(photos))`` bytes).  No CUDA call; returns the number of tiles."""
    l = _lib.lib()
    n = len(photos)
    docs = (_lib.UnwarpDoc * n)(*[_lib.UnwarpDoc(p.data_ptr(), o.data_ptr(), p.shape[0], p.shape[1]) for p, o in zip(photos, outs)])
    tiles = C_longlong(0)
    _lib.check(l.dvd_unwarp_u8_plan(docs if n else None, n, C, mh, mw, affine, _lib.ptr(table_host), table_host.numel(), byref(tiles)),
               "dvd_unwarp_u8_plan")
    return tiles.value


def table_bytes(max_docs: int) -> int:
    """bytes of a mixed-size unwarp table for up to `max_docs` documents"""
    return _lib.lib().dvd_unwarp_table_bytes(max_docs)


def sized_table_bytes(max_docs: int) -> int:
    """bytes of a sized unwarp table for up to `max_docs` documents"""
    return _lib.lib().dvd_unwarp_sized_table_bytes(max_docs)


def plan_sized(table_host: torch.Tensor, photos, outs, mh: int, mw: int, supersample=0, affine: float = AFFINE, C: int = 3):
    """Plans a sized uint8 HWC batch (document i: photos[i] [H,W,C] -> outs[i] [Ho,Wo,C], device tensors) into the host tensor
    `table_host` (pinned uint8, at least ``sized_table_bytes(len(photos))`` bytes).  `supersample`: 0 (auto) or 1..8, one for all
    documents or a list.  No CUDA call; returns (tiles, the factor chosen for each document)."""
    l = _lib.lib()
    n = len(photos)
    ss = list(supersample) if isinstance(supersample, (list, tuple)) else [supersample] * n
    docs = (_lib.SizedUnwarpDoc * max(n, 1))(*[_lib.SizedUnwarpDoc(p.data_ptr(), o.data_ptr(), p.shape[0], p.shape[1], o.shape[0],
                                                                   o.shape[1], s, 0) for p, o, s in zip(photos, outs, ss)])
    tiles = C_longlong(0)
    chosen = (C_int32 * max(n, 1))()
    _lib.check(l.dvd_unwarp_u8_sized_plan(docs if n else None, n, C, mh, mw, affine, _lib.ptr(table_host), table_host.numel(),
                                          byref(tiles), chosen), "dvd_unwarp_u8_sized_plan")
    return tiles.value, list(chosen)[:n]


def supersample_arg(supersample) -> int:
    """"auto" -> 0 (the planner's choice), 1..8 -> itself; anything else is a ValueError"""
    if isinstance(supersample, str) and supersample == "auto":
        return 0
    if isinstance(supersample, bool) or not isinstance(supersample, int) or not 1 <= supersample <= 8:
        raise ValueError(f"supersample must be 'auto' or an integer in 1..8, got {supersample!r}")
    return supersample


def size_arg(size, what: str = "size") -> tuple:
    """(Ho, Wo) with positive integers, else a ValueError"""
    if (not isinstance(size, (tuple, list)) or len(size) != 2
            or not all(isinstance(v, int) and not isinstance(v, bool) and v >= 1 for v in size)):
        raise ValueError(f"{what} must be (Ho, Wo) with positive integers, got {size!r}")
    return int(size[0]), int(size[1])


def _dewarp_planned(map64: torch.Tensor, photos, outs, sized: bool, supersample: int, affine: float):
    """one launch over a planned table: photos[i] -> outs[i] with map row i; the sized launch when `sized`, else the mixed-size one"""
    if not photos:
        return
    Cc, mh, mw = photos[0].shape[2], map64.shape[2], map64.shape[3]
    if sized:
        nbytes, launch = sized_table_bytes(len(photos)), "dvd_unwarp_u8_sized"
        plan = lambda host: plan_sized(host, photos, outs, mh, mw, supersample, affine, Cc)
    else:
        nbytes, launch = table_bytes(len(photos)), "dvd_unwarp_u8_mixed"
        plan = lambda host: plan_mixed(host, photos, outs, mh, mw, affine, Cc)
    table = _lib.PlannedTable(nbytes, map64.device).upload(plan)
    _lib.check(getattr(_lib.lib(), launch)(_lib.ptr(table), Cc, _lib.ptr(map64), _lib.stream_ptr()), launch)


def _dewarp_mixed(map64: torch.Tensor, photos, affine: float, size=None, supersample: int = 0) -> list:
    photos = list(photos)
    if map64.dim() != 4 or map64.shape[0] != len(photos):
        raise ValueError(f"map64 {tuple(map64.shape)} does not have one row per photo ({len(photos)})")
    for i, p in enumerate(photos):
        if p.dtype != torch.uint8 or p.dim() != 3 or not p.is_contiguous() or p.device != map64.device:
            raise ValueError(f"photo {i}: a list of photos takes contiguous uint8 HWC tensors on {map64.device}, got "
                             f"{p.dtype} {tuple(p.shape)} on {p.device}")
        if p.shape[2] != photos[0].shape[2]:
            raise ValueError(f"photo {i} has {p.shape[2]} channels, photo 0 has {photos[0].shape[2]}")
    if size is None:
        outs = [torch.empty_like(p) for p in photos]
    else:
        per_photo = isinstance(size, list) and (not size or isinstance(size[0], (tuple, list)))
        sizes = list(size) if per_photo else [size] * len(photos)
        if len(sizes) != len(photos):
            raise ValueError(f"size: {len(sizes)} sizes for {len(photos)} photos")
        sizes = [size_arg(s, f"size of photo {i}") for i, s in enumerate(sizes)]
        outs = [torch.empty((Ho, Wo, p.shape[2]), dtype=torch.uint8, device=p.device) for p, (Ho, Wo) in zip(photos, sizes)]
    _dewarp_planned(map64, photos, outs, size is not None, supersample, affine)
    return outs


@torch.no_grad()
def dewarp_fullres(map64: torch.Tensor, photo, out: torch.Tensor | None = None, out_uint8: bool = False,
                   affine: float = AFFINE, size=None, supersample="auto"):
    """map64 [B,2,h,w] fp32 displacement (sampler output); photo either fp32 NCHW [B,C,H,W] (values
    0..255, the reference's ``source_image_ori``) or uint8 NHWC [B,H,W,C].
    Returns fp32 NCHW, or uint8 NHWC (truncated like ``.astype(np.uint8)``) when ``out_uint8`` / uint8 input.

    ``photo`` may also be a list / tuple of B uint8 HWC device tensors [H_i,W_i,C] of different sizes: one launch dewarps them
    all (photo i with map row i) and a list of B new uint8 HWC tensors is returned (``out`` / ``out_uint8`` do not apply).

    ``size=(Ho, Wo)`` (uint8 photos only) writes the page at Ho x Wo instead of the photo's size, in one launch: a uint8 NHWC
    batch gives [B,Ho,Wo,C] (into ``out`` if given), a list gives a list, and a list takes either one size for every photo or a
    list of one (Ho, Wo) per photo.  ``supersample`` ("auto" or 1..8) is the factor s: each output pixel is the mean of an
    s x s block of the reference chain evaluated at s*Ho x s*Wo, truncated; "auto" is min(8, max(1, ceil(H/Ho), ceil(W/Wo))).
    ``size=None`` is the photo-size output above."""
    _chk(map64, "map64")
    ss = supersample_arg(supersample)
    if isinstance(photo, (list, tuple)):
        if out is not None:
            raise ValueError("dewarp_fullres: `out` does not apply to a list of photos")
        map64 = map64.float().contiguous()
        with torch.cuda.device(map64.device):
            return _dewarp_mixed(map64, photo, affine, size, ss)
    _chk(photo, "photo")
    if size is not None:
        if photo.dtype != torch.uint8 or photo.dim() != 4:
            raise ValueError(f"dewarp_fullres: size= takes uint8 NHWC photos, got {photo.dtype} {tuple(photo.shape)}")
        Ho, Wo = size_arg(size)
        map64 = map64.float().contiguous()
        photo = photo.contiguous()
        B, H, W, Cc = photo.shape
        if map64.dim() != 4 or map64.shape[0] != B or photo.device != map64.device:
            raise ValueError(f"map64 {tuple(map64.shape)} on {map64.device} does not have one row per photo ({B}) on {photo.device}")
        if out is None:
            out = torch.empty((B, Ho, Wo, Cc), dtype=torch.uint8, device=photo.device)
        elif out.dtype != torch.uint8 or tuple(out.shape) != (B, Ho, Wo, Cc) or not out.is_contiguous() or out.device != photo.device:
            raise ValueError(f"out must be a contiguous uint8 tensor {(B, Ho, Wo, Cc)} on {photo.device}, got {out.dtype} "
                             f"{tuple(out.shape)}")
        with torch.cuda.device(photo.device):
            _dewarp_planned(map64, list(photo.unbind(0)), list(out.unbind(0)), True, ss, affine)
        return out
    map64 = map64.float().contiguous()
    l = _lib.lib()
    B, _, mh, mw = map64.shape
    with torch.cuda.device(photo.device):
        st = _lib.stream_ptr()
        if photo.dtype == torch.uint8:
            photo = photo.contiguous()
            Bp, H, W, Cc = photo.shape
            assert Bp == B
            out = torch.empty_like(photo) if out is None else out
            _lib.check(l.dvd_unwarp_u8(_lib.ptr(photo), _lib.ptr(map64), _lib.ptr(out), B, Cc, H, W, mh, mw, affine, st), "dvd_unwarp_u8")
            return out
        photo = photo.float().contiguous()
        Bp, Cc, H, W = photo.shape
        assert Bp == B
        if out_uint8:
            out = torch.empty((B, H, W, Cc), dtype=torch.uint8, device=photo.device) if out is None else out
            _lib.check(l.dvd_unwarp_f32_u8(_lib.ptr(photo), _lib.ptr(map64), _lib.ptr(out), B, Cc, H, W, mh, mw, affine, st),
                       "dvd_unwarp_f32_u8")
            return out
        out = torch.empty_like(photo) if out is None else out
        _lib.check(l.dvd_unwarp_f32(_lib.ptr(photo), _lib.ptr(map64), _lib.ptr(out), B, Cc, H, W, mh, mw, affine, st), "dvd_unwarp_f32")
        return out


@torch.no_grad()
def fullres_grid(map64: torch.Tensor, H: int, W: int, affine: float = AFFINE) -> torch.Tensor:
    """evaluation.py:301-306 materialised ([B,2,H,W]); used by parity tests and by callers that still want the grid."""
    _chk(map64, "map64")
    map64 = map64.float().contiguous()
    B, _, mh, mw = map64.shape
    grid = torch.empty((B, 2, H, W), dtype=torch.float32, device=map64.device)
    with torch.cuda.device(map64.device):
        _lib.check(_lib.lib().dvd_fullres_grid_f32(_lib.ptr(map64), _lib.ptr(grid), B, H, W, mh, mw, affine, _lib.stream_ptr()),
                   "dvd_fullres_grid_f32")
    return grid
