"""The call a user makes: photo(s) + conditioning in, dewarped image(s) out.

``DewarpPipeline`` is the hot part of the reference's per-document loop
(train_settings/dvd/evaluation.py:245-268 sampling, :300-306 upsample/affine, :317-318 unwarp) for
a fixed batch of ``docs`` documents per call.  Everything between the inputs and the dewarped
image runs in libdvd_b200; torch only owns the buffers and the stream.

With ``max_pixels=P`` the pipeline takes photos of different sizes in one batch (mixed-size mode): ``photo_u8`` is then a list of
uint8 HWC tensors whose pixel counts sum to at most P, the results are a list of uint8 HWC images, and one unwarp launch, captured
once per set of buffers, serves every composition of sizes.

With ``out_size`` the dewarped pages come out at a requested size instead of the photo's: a ``(Ho, Wo)`` tuple, or a callable
``(H, W) -> (Ho, Wo)`` evaluated per photo.  The unwarp step is then the sized launch (supersampled when shrinking), so only the
smaller pages are written and downloaded.

With ``y512_from_photo=True`` the denoiser's 512x512 input is computed from ``photo_u8`` on the GPU (the reference loader's
``cv2.resize(photo, (512, 512), INTER_LINEAR) / 255``, byte for byte) by one launch at the head of the sampling graph; the input
dicts then carry no ``y512`` and the host path uploads none.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import torch

from . import _lib
from .model import DiT
from .inputs import launch_y512, plan_y512, table_bytes as y512_table_bytes
from .sampler import create_gaussian_diffusion
from .unwarp import AFFINE, plan_mixed, plan_sized, size_arg, sized_table_bytes, supersample_arg, table_bytes


class DewarpPipeline:
    def __init__(self, model: DiT, diffusion_steps: int = 3, n_batch: int = 2, docs: int = 1, height: int = 1500, width: int = 2000,
                 noise_schedule: str = "cosine", precision: str | None = None, max_pixels: int | None = None, out_size=None,
                 supersample="auto", max_out_pixels: int | None = None, y512_from_photo: bool = False):
        self.model, self.docs, self.n_batch, self.H, self.W = model, docs, n_batch, height, width
        # y512 computed from photo_u8 by the first launch of the sampling graph instead of supplied by the caller
        self.y512_from_photo = bool(y512_from_photo)
        self._input_keys = self.SAMPLING_KEYS[1:] if self.y512_from_photo else self.SAMPLING_KEYS
        self._sampling_keys = self.SAMPLING_KEYS + ("prep",) if self.y512_from_photo else self.SAMPLING_KEYS
        self._sampling = self._enqueue_prep_sampling if self.y512_from_photo else self._enqueue_sampling
        self.max_pixels = max_pixels
        if max_pixels is not None and max_pixels < 1:
            raise ValueError(f"max_pixels must be positive, got {max_pixels}")
        # output size (None: the photo's).  Fixed-size mode: one (Ho, Wo) for the batch; mixed-size mode: per photo, into an arena
        # of max_out_pixels (default max_pixels)
        self.out_size, self.supersample = out_size, supersample_arg(supersample)
        if out_size is not None and not callable(out_size):
            size_arg(out_size, "out_size")
        if max_out_pixels is not None and (out_size is None or max_pixels is None or max_out_pixels < 1):
            raise ValueError("max_out_pixels takes a positive count and applies to mixed-size mode (max_pixels) with out_size")
        self.max_out_pixels = max_out_pixels if max_out_pixels is not None else max_pixels
        self.HWo = self._out_hw(height, width) if out_size is not None and max_pixels is None else (height, width)
        self.precision = precision or model.precision
        self.dev = model.device
        if self.dev.type != "cuda":
            raise RuntimeError("DewarpPipeline needs the model on a CUDA device (no CPU path)")
        self.diffusion = create_gaussian_diffusion(steps=diffusion_steps, noise_schedule=noise_schedule, predict_xstart=True,
                                                   rescale_timesteps=True, rescale_learned_sigmas=True, timestep_respacing="")
        self.lib = _lib.lib()
        # the unwarp: the batched fixed-size launch, or one launch over a table planned per batch (mixed size, out_size)
        if out_size is not None:
            self._plan_unwarp = lambda host, photos, outs: plan_sized(host, photos, outs, 64, 64, self.supersample)
            self._unwarp_launch, self._unwarp_bytes = "dvd_unwarp_u8_sized", sized_table_bytes(docs)
        elif max_pixels is not None:
            self._plan_unwarp = lambda host, photos, outs: plan_mixed(host, photos, outs, 64, 64)
            self._unwarp_launch, self._unwarp_bytes = "dvd_unwarp_u8_mixed", table_bytes(docs)
        else:
            self._plan_unwarp = None
        with torch.cuda.device(self.dev):
            self._bind_engine()
            z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=self.dev)
            # mixed-size mode: photos and outputs live in byte arenas, each document at a 16-byte aligned offset
            img = (docs, height, width, 3) if max_pixels is None else (3 * max_pixels + 16 * docs,)
            oimg = (docs,) + self.HWo + (3,) if max_pixels is None else (3 * self.max_out_pixels + 16 * docs,)
            self.buf = {"y512": z(docs, 3, 512, 512), "mask_cat": z(docs, 1, 512, 512), "mask_y512": z(docs, 384, 64, 64),
                        "line_msk": z(docs, 64, 64, 64), "x_T": z(docs * n_batch, 2, 64, 64),
                        "photo_u8": z(*img, dt=torch.uint8)}
            self.init_flow0 = z(docs, 2, 64, 64)                       # evaluation.py:180 (use_init_flow=False)
            self.map64 = z(docs, 2, 64, 64)
            self.out_u8 = z(*oimg, dt=torch.uint8)
            self._device_tables = self._planned_tables()              # run_device's
        self.h2d_bytes = sum(v.numel() * v.element_size() for k, v in self.buf.items() if k in self._input_keys + ("photo_u8",))
        self.d2h_bytes = self.out_u8.numel()
        self.use_graph = os.environ.get("DVD_NO_GRAPH", "0") != "1"
        self.kernel_launches = 0           # kernels of libdvd_b200 launched (or replayed) through this pipeline
        self._slots = None                 # double-buffered host I/O state (submit_host / wait)

    def _bind_engine(self):
        """(Re)binds the engine, conditioning tables and graphs to the model's CURRENT packed weights: load_state_dict() / .to()
        on the model replace them, and a pipeline that kept serving the old ones would silently use stale weights."""
        self.eng = self.model.engine(self.docs, self.n_batch, self.precision)
        self._packed = self.eng.packed
        self.t_scaled, t_emb, self.a, self.b = self.diffusion._plan()
        self.tables = self.eng.tables(t_emb)
        self._graphs = {}

    def _check_weights(self):
        if self.model.device != self.dev:
            raise RuntimeError("DewarpPipeline: the model was moved to another device; build a new pipeline")
        if self.model.packed() is not self._packed:
            with torch.cuda.device(self.dev):
                self._bind_engine()

    def _planned_tables(self) -> dict:
        """the host-planned launch tables of one batch in flight: "unwarp" (mixed size or out_size) and "prep" (y512_from_photo)"""
        tables = {}
        if self._plan_unwarp is not None:
            tables["unwarp"] = _lib.PlannedTable(self._unwarp_bytes, self.dev)
        if self.y512_from_photo:
            tables["prep"] = _lib.PlannedTable(y512_table_bytes(self.docs), self.dev)
        return tables

    # ---- device-resident inputs: dict with y512, mask_cat, mask_y512, line_msk, x_T, photo_u8 (all on self.dev)
    def _enqueue_sampling(self, d: dict):
        """static conditioning -> S-step DDIM loop -> hypothesis mean (map64), on the current stream."""
        self.eng.static_forward(d["y512"], d["mask_cat"], d["mask_y512"], d["line_msk"])
        self.eng.sample(d["x_T"], self.init_flow0, self.tables, self.t_scaled, self.a, self.b, None, self.map64)

    def _enqueue_prep_sampling(self, d: dict):
        """y512 from the photos planned into the device table d["prep"], then the sampling above."""
        launch_y512(d["prep"], d["y512"])
        self._enqueue_sampling(d)

    def _enqueue_unwarp(self, d: dict):
        """fused upsample + affine + bilinear unwarp of the full-resolution photos d["photo_u8"] into d["out_u8"], on the current
        stream."""
        _lib.check(self.lib.dvd_unwarp_u8(_lib.ptr(d["photo_u8"]), _lib.ptr(self.map64), _lib.ptr(d["out_u8"]), self.docs, 3,
                                          self.H, self.W, 64, 64, AFFINE, _lib.stream_ptr()), "dvd_unwarp_u8")

    def _enqueue_unwarp_table(self, d: dict):
        """mixed-size or sized unwarp of the batch planned into the device table d["table"] (one launch whatever the composition)."""
        fn = self._unwarp_launch
        _lib.check(getattr(self.lib, fn)(_lib.ptr(d["table"]), 3, _lib.ptr(self.map64), _lib.stream_ptr()), fn)

    def _sample(self, d: dict, photos, tables: dict):
        """the sampling graph on the current stream; with y512_from_photo its first launch reads a y512 table planned from `photos`"""
        if self.y512_from_photo:
            d = dict(d, prep=tables["prep"].upload(lambda host: plan_y512(host, photos)))
        self._run("sampling", d, self._sampling_keys, self._sampling)

    def _unwarp(self, photos, outs, tables: dict):
        """the unwarp graph on the current stream: photos -> outs with the rows of map64"""
        if self._plan_unwarp is None:
            self._run("unwarp", {"photo_u8": photos, "out_u8": outs}, ("photo_u8", "out_u8"), self._enqueue_unwarp)
        else:
            table = tables["unwarp"].upload(lambda host: self._plan_unwarp(host, photos, outs))
            self._run("unwarp", {"table": table}, ("table",), self._enqueue_unwarp_table)

    def _out_hw(self, H: int, W: int) -> tuple:
        """output size of an H x W photo"""
        return size_arg(self.out_size(H, W) if callable(self.out_size) else self.out_size, f"out_size for a {H}x{W} photo")

    def _place(self, buf: torch.Tensor, docs):
        """a batch in `buf`: fixed-size mode, the [docs,...] buffer itself; mixed-size mode, one view per document (a tensor or a
        shape) packed into the arena `buf`"""
        return buf if self.max_pixels is None else self._arena_views(buf, docs)

    def _outputs(self, buf: torch.Tensor, photos):
        """where the pages of a batch go in `buf`; in mixed-size mode with out_size, their shapes hold at most max_out_pixels"""
        if self.max_pixels is None or self.out_size is None:
            return self._place(buf, photos)
        shapes = [self._out_hw(p.shape[0], p.shape[1]) + (3,) for p in photos]
        px = sum(Ho * Wo for Ho, Wo, _ in shapes)
        if px > self.max_out_pixels:
            raise ValueError(f"the batch's outputs have {px} pixels, more than max_out_pixels={self.max_out_pixels}")
        return self._arena_views(buf, shapes)

    def _check_inputs(self, d: dict, on_device: bool):
        """Validates the inputs of one batch and returns its photos.  A host dict carries 1..docs photos (fixed-size mode: docs) on
        the CPU, a device dict exactly docs photos and contiguous fp32 sampling inputs on the pipeline's device; the other inputs
        have one row per photo (x_T n_batch rows)."""
        if self.y512_from_photo and "y512" in d:
            raise ValueError("this pipeline computes y512 from photo_u8 (y512_from_photo=True); do not pass y512")
        photos = self._check_photos(d["photo_u8"], self.dev if on_device else torch.device("cpu"), self.docs if on_device else 1)
        n = len(photos)
        for k in self._input_keys:
            t = d[k]
            want = (n * self.n_batch if k == "x_T" else n,) + tuple(self.buf[k].shape[1:])
            if tuple(t.shape) != want:
                raise ValueError(f"{k}: expected shape {want} for {n} photos, got {tuple(t.shape)}")
            if on_device and (t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.dev):
                raise ValueError(f"{k}: expected a contiguous float32 tensor on {self.dev}, got {t.dtype} on {t.device}")
        return photos

    def _check_photos(self, photos, device: torch.device, lo: int):
        """Validates the photos of a batch on `device`: fixed-size mode, one contiguous uint8 tensor [docs,H,W,3]; mixed-size mode,
        lo..docs uint8 HWC RGB tensors with at most max_pixels in all (returned as a list)."""
        if self.max_pixels is None:
            want = (self.docs, self.H, self.W, 3)
            if (not isinstance(photos, torch.Tensor) or photos.dtype != torch.uint8 or tuple(photos.shape) != want
                    or not photos.is_contiguous() or photos.device != device):
                raise ValueError(f"photo_u8: expected a contiguous uint8 tensor {want} on {device}, got "
                                 f"{getattr(photos, 'dtype', type(photos))} {tuple(getattr(photos, 'shape', ()))} "
                                 f"on {getattr(photos, 'device', None)}")
            return photos
        if not isinstance(photos, (list, tuple)):
            raise ValueError("mixed-size mode (max_pixels) takes photo_u8 as a list of uint8 HWC tensors")
        if not lo <= len(photos) <= self.docs:
            raise ValueError(f"{len(photos)} photos: this call takes {lo}..{self.docs}" if lo < self.docs else
                             f"{len(photos)} photos: this call takes exactly {self.docs}")
        for i, p in enumerate(photos):
            if not isinstance(p, torch.Tensor) or p.dtype != torch.uint8 or p.dim() != 3 or p.shape[2] != 3:
                raise ValueError(f"photo {i}: expected a uint8 HWC tensor with 3 channels, got "
                                 f"{getattr(p, 'dtype', type(p))} {tuple(getattr(p, 'shape', ()))}")
            if not p.is_contiguous():
                raise ValueError(f"photo {i} is not contiguous")
            if p.device != device:
                raise ValueError(f"photo {i} is on {p.device}, this call takes photos on {device}")
        px = sum(p.shape[0] * p.shape[1] for p in photos)
        if px > self.max_pixels:
            raise ValueError(f"the batch has {px} pixels, more than max_pixels={self.max_pixels}")
        return list(photos)

    @staticmethod
    def _arena_views(arena: torch.Tensor, photos) -> list:
        """one [H,W,3] view per photo (tensor or shape), packed at 16-byte aligned offsets"""
        views, off = [], 0
        for p in photos:
            shape = tuple(p.shape) if isinstance(p, torch.Tensor) else tuple(p)
            n = shape[0] * shape[1] * shape[2]
            views.append(arena[off:off + n].view(shape))
            off = (off + n + 15) & ~15
        return views

    def _graph(self, which: str, d: dict, keys, fn):
        """CUDA graph of `fn(d)` for this set of input buffers (captured once, replayed afterwards)."""
        key = (which,) + tuple(d[k].data_ptr() for k in keys)
        if key not in self._graphs:
            fn(d)                                                  # eager warm-up (function attributes, driver entry points)
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            n0 = self.lib.dvd_launch_count(0)
            with torch.cuda.graph(g):
                fn(d)
            if len(self._graphs) >= 16:
                self._graphs.pop(next(iter(self._graphs)))
            self._graphs[key] = (g, self.lib.dvd_launch_count(0) - n0, d)
        return self._graphs[key]

    def _run(self, which: str, d: dict, keys, fn):
        if not self.use_graph:
            n0 = self.lib.dvd_launch_count(0)
            fn(d)
            self.kernel_launches += self.lib.dvd_launch_count(0) - n0
            return
        g, n, _ = self._graph(which, d, keys, fn)
        g.replay()
        self.kernel_launches += n

    SAMPLING_KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")

    def run_device(self, d: dict):
        """The ~230 kernel launches of one batch are captured once per set of input buffers into two CUDA graphs (sampling,
        unwarp) and replayed (the library never allocates or synchronises, so every entry point is capturable).  Returns the
        device output, overwritten by the next call.

        Mixed-size mode: d["photo_u8"] is a list of exactly `docs` uint8 HWC photos on the pipeline's device (read in place);
        returns a list of views into the device output arena."""
        self._check_weights()
        photos = self._check_inputs(d, on_device=True)
        with torch.cuda.device(self.dev):
            outs = self._outputs(self.out_u8, photos)
            if self.y512_from_photo:
                d = dict(d, y512=self.buf["y512"])
            self._sample(d, photos, self._device_tables)
            self._unwarp(photos, outs, self._device_tables)
        return outs

    # ---- pinned-host inputs -> host uint8 image (H2D and D2H inside the call)
    def _make_slots(self):
        """Two sets of device input / output buffers, planned tables + copy streams: the uploads of batch i+1 and the download of
        batch i run underneath the kernels of the batch in between (the kernels themselves stay on the caller's stream, one batch
        at a time)."""
        self._h2d = torch.cuda.Stream(device=self.dev)
        self._d2h = torch.cuda.Stream(device=self.dev)
        self._slots = []
        for _ in range(2):
            buf = {k: torch.empty_like(v) for k, v in self.buf.items()}
            buf["out_u8"] = torch.empty_like(self.out_u8)
            self._slots.append({"buf": buf, "out_host": torch.empty(self.out_u8.shape, dtype=torch.uint8, pin_memory=True),
                                "tables": self._planned_tables(), "result": None, "used": False, "ev_in": torch.cuda.Event(),
                                "ev_photo": torch.cuda.Event(), "ev_done": torch.cuda.Event(), "ev_out": torch.cuda.Event()})
        self._submitted = 0

    def submit_host(self, h: dict) -> int:
        """Enqueue one batch (pinned host inputs) without waiting for it; returns a ticket for `wait`.  At most two batches may be
        outstanding (a ticket must be waited for before the second-next submit).  The photo is only needed by the last kernel, so
        its upload also runs underneath this batch's own sampling.

        Mixed-size mode: h["photo_u8"] is a list of 1..docs uint8 HWC host photos and the other inputs have that many documents
        (x_T that many times n_batch); document slots past the list keep their earlier inputs, are sampled and not unwarped."""
        self._check_weights()
        photos = self._check_inputs(h, on_device=False)
        with torch.cuda.device(self.dev):
            if self._slots is None:
                self._make_slots()
            main = torch.cuda.current_stream()
            ticket = self._submitted
            s = self._slots[ticket % 2]
            buf = s["buf"]
            photo_dev, out_dev = self._place(buf["photo_u8"], photos), self._outputs(buf["out_u8"], photos)
            self._submitted += 1
            with torch.cuda.stream(self._h2d):
                if s["used"]:
                    self._h2d.wait_event(s["ev_done"])             # the kernels of batch ticket-2 have read this slot's inputs
                for k in self._input_keys:
                    buf[k][:h[k].shape[0]].copy_(h[k], non_blocking=True)
                s["ev_in"].record()
                if self.max_pixels is None:
                    photo_dev.copy_(photos, non_blocking=True)
                else:
                    for dst, src in zip(photo_dev, photos):
                        dst.copy_(src, non_blocking=True)
                s["ev_photo"].record()
            main.wait_event(s["ev_photo"] if self.y512_from_photo else s["ev_in"])      # y512 from the photo: sampling reads it
            if s["used"]:
                main.wait_event(s["ev_out"])                       # the download of batch ticket-2 has read this slot's output
            self._sample(buf, photo_dev, s["tables"])
            main.wait_event(s["ev_photo"])
            self._unwarp(photo_dev, out_dev, s["tables"])
            s["ev_done"].record(main)
            end = out_dev[-1].data_ptr() - buf["out_u8"].data_ptr() + out_dev[-1].numel()       # through the batch's last page
            with torch.cuda.stream(self._d2h):
                self._d2h.wait_event(s["ev_done"])
                s["out_host"].view(-1)[:end].copy_(buf["out_u8"].view(-1)[:end], non_blocking=True)
                s["ev_out"].record()
            s["result"] = self._place(s["out_host"], out_dev)
            s["used"] = True
        return ticket

    def wait(self, ticket: int):
        """Block until the batch of `ticket` is on the host; the returned pinned tensor (mixed-size mode: list of views into a
        pinned arena) is reused by the second-next submit."""
        s = self._slots[ticket % 2]
        s["ev_out"].synchronize()
        return s["result"]

    def run_host(self, h: dict):
        """Synchronous form: host inputs in, host uint8 image(s) out."""
        return self.wait(self.submit_host(h))

    # ---- measurement helpers used by bench.py
    def profile_kernels(self, d: dict, iters: int = 5, with_unwarp: bool = True) -> dict:
        """CUDA-event timing (on the launch stream, L2 flushed between runs) of the kernel classes inside a real step, and of
        the unwarp kernel; returns the roofline objects of the bench JSON line."""
        peaks_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
        try:
            peaks = json.load(open(peaks_path)); which = "measured"
        except Exception:
            peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}; which = "fallback"
        with torch.cuda.device(self.dev):
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
            ms, fl, ln, fx = (C.c_double * 3)(), (C.c_double * 3)(), (C.c_longlong * 3)(), (C.c_double * 3)()
            tot_ms, tot = [0.0, 0.0, 0.0], 0.0
            for it in range(iters):
                flush.fill_(it)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                self.lib.dvd_profile_begin()
                e0.record()
                self.eng.static_forward(d["y512"], d["mask_cat"], d["mask_y512"], d["line_msk"])
                self.eng.sample(d["x_T"], self.init_flow0, self.tables, self.t_scaled, self.a, self.b, None, self.map64)
                e1.record()
                _lib.check(self.lib.dvd_profile_end(ms, fl, ln, fx), "dvd_profile_end")
                if it == 0:
                    continue                                        # warm-up
                tot += e0.elapsed_time(e1)
                for c in range(3):
                    tot_ms[c] += ms[c]
            n = iters - 1
            share = {"gemm": tot_ms[0] / tot, "attention": tot_ms[1] / tot, "pyramid_conv": tot_ms[2] / tot,
                     "other": 1.0 - sum(tot_ms) / tot, "denoiser_ms_per_step": tot / n}
            gemm_tf = fl[0] / (tot_ms[0] / n * 1e-3) / 1e12 if tot_ms[0] > 0 else 0.0
            attn_tf = fl[1] / (tot_ms[1] / n * 1e-3) / 1e12 if tot_ms[1] > 0 else 0.0
            try:
                traffic = json.load(open(os.path.join(os.path.dirname(peaks_path), "profiles", "r2_traffic.json")))
            except Exception:
                traffic = {}
            tensor_mode = self.precision in ("bf16", "bf16x3")
            exec_tf = fx[0] / (tot_ms[0] / n * 1e-3) / 1e12 if tot_ms[0] > 0 else 0.0
            peak_tf = peaks["bf16_tflops_sustained"] if tensor_mode else 72.0      # fp32 FFMA: 148 SM x 128 FMA x 2 x 1.9 GHz
            roof = {"kernel": "k_gemm_pair: dense GEMM (all linear layers of one step batch)", "bound": "tensor", "achieved": gemm_tf,
                    "peak": peak_tf, "unit": "TFLOP/s", "frac": gemm_tf / peak_tf,
                    "traffic": (traffic.get("gemm_dominant") if self.precision == "bf16x3" else None),
                    "launches_per_step": int(ln[0]), "gflop_per_step": fl[0] / 1e9, "attention_tflops": attn_tf,
                    "attention_gflop_per_step": fl[1] / 1e9,
                    # achieved / frac count ALGORITHMIC flops (2 M N K).  The split-precision mode executes three tensor-core passes per
                    # k-step to be fp32-accurate (two in the decoder's q|k|v GEMM), so its tensor pipe does `mma_passes` x that work on
                    # average: frac_executed is the pipe's own load.
                    "mma_passes": round(fx[0] / fl[0], 3) if fl[0] > 0 else 1, "executed_tflops": exec_tf, "frac_executed": exec_tf / peak_tf,
                    "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (%s)" % which) if tensor_mode else "nominal fp32 FFMA"}
            if not with_unwarp:
                return {"roofline": roof, "share": share}
            # unwarp: fp32 contract (24 B/px) and the uint8 variant actually used end to end (6 B/px).  20 launches replayed from one
            # CUDA graph (no host time between launches) over rotating buffer pairs whose total exceeds the L2, so every launch
            # reads its photo from HBM.
            photo_f = d["photo_u8"].permute(0, 3, 1, 2).float().contiguous()
            px = self.docs * self.H * self.W
            st = _lib.stream_ptr()

            # The map sampled with random-init weights is white noise (neighbouring coarse-map cells differ by hundreds of pixels), which
            # no document produces; the roofline is therefore quoted on a smooth synthetic warp (bicubic-upsampled 8x8 field, amplitude
            # 0.02 = ~20% local shear) and the noise map's time is reported next to it.
            gen = torch.Generator(device="cpu").manual_seed(3005)
            smooth = torch.nn.functional.interpolate(torch.randn((1, 2, 8, 8), generator=gen) * 0.02, size=(64, 64), mode="bicubic",
                                                     align_corners=True).clamp(-1, 1).repeat(self.docs, 1, 1, 1).contiguous().to(self.dev)

            def time_unwarp(src, fn_name, map64, n_launch=20):
                per = 2 * src.numel() * src.element_size()
                nbuf = max(2, (300 << 20) // per + 1)
                ins = [src.clone() for _ in range(nbuf)]
                outs = [torch.empty_like(src) for _ in range(nbuf)]
                fn = getattr(self.lib, fn_name)

                def launch(i):
                    _lib.check(fn(_lib.ptr(ins[i % nbuf]), _lib.ptr(map64), _lib.ptr(outs[i % nbuf]), self.docs, 3, self.H, self.W,
                                  64, 64, AFFINE, _lib.stream_ptr()), fn_name)
                for i in range(nbuf):
                    launch(i)
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    for i in range(n_launch):
                        launch(i)
                graph.replay(); torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); graph.replay(); e1.record(); e1.synchronize()
                return e0.elapsed_time(e1) / n_launch
            t32 = time_unwarp(photo_f, "dvd_unwarp_f32", smooth)
            t8 = time_unwarp(d["photo_u8"], "dvd_unwarp_u8", smooth)
            t32_noise = time_unwarp(photo_f, "dvd_unwarp_f32", self.map64)
            t8_noise = time_unwarp(d["photo_u8"], "dvd_unwarp_u8", self.map64)
            gb32, gb8 = 24.0 * px / 1e9, 6.0 * px / 1e9
            ru = {"kernel": "k_unwarp_tma fp32 NCHW (24 B/px)", "map": "smooth synthetic warp, amplitude 0.02", "bound": "hbm", "achieved": gb32 / (t32 * 1e-3), "peak": peaks["hbm_gbs"],
                  "unit": "GB/s", "frac": gb32 / (t32 * 1e-3) / peaks["hbm_gbs"],
                  "traffic": (traffic.get("unwarp_f32_1500x2000") if (self.H, self.W) == (1500, 2000) else None), "ms": t32,
                  "u8_variant": {"achieved": gb8 / (t8 * 1e-3), "frac": gb8 / (t8 * 1e-3) / peaks["hbm_gbs"], "ms": t8, "bytes_per_px": 6},
                  "random_init_map": {"note": "the map sampled with random-init weights is white noise", "ms_f32": t32_noise, "ms_u8": t8_noise},
                  "peak_source": "MEASURED_PEAKS.json hbm_gbs (%s)" % which}
        return {"roofline": roof, "roofline_unwarp": ru, "share": share}
