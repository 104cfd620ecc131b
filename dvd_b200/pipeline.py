"""The call a user makes: photo(s) + conditioning in, dewarped image(s) out.

``DewarpPipeline`` is the hot part of the reference's per-document loop
(train_settings/dvd/evaluation.py:245-268 sampling, :300-306 upsample/affine, :317-318 unwarp) for
a fixed batch of ``docs`` documents per call.  Everything between the inputs and the dewarped
image runs in libdvd_b200; torch only owns the buffers and the stream.

With ``max_pixels=P`` the pipeline takes photos of different sizes in one batch (mixed-size mode): ``photo_u8`` is then a list of
uint8 HWC tensors whose pixel counts sum to at most P, the results are a list of uint8 HWC images, and one unwarp launch, captured
once per set of buffers, serves every composition of sizes.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import torch

from . import _lib
from .model import DiT
from .sampler import create_gaussian_diffusion
from .unwarp import AFFINE, plan_mixed, table_bytes


class DewarpPipeline:
    def __init__(self, model: DiT, diffusion_steps: int = 3, n_batch: int = 2, docs: int = 1, height: int = 1500, width: int = 2000,
                 noise_schedule: str = "cosine", precision: str | None = None, max_pixels: int | None = None):
        self.model, self.docs, self.n_batch, self.H, self.W = model, docs, n_batch, height, width
        self.max_pixels = max_pixels
        if max_pixels is not None and max_pixels < 1:
            raise ValueError(f"max_pixels must be positive, got {max_pixels}")
        self.precision = precision or model.precision
        self.dev = model.device
        if self.dev.type != "cuda":
            raise RuntimeError("DewarpPipeline needs the model on a CUDA device (no CPU path)")
        self.diffusion = create_gaussian_diffusion(steps=diffusion_steps, noise_schedule=noise_schedule, predict_xstart=True,
                                                   rescale_timesteps=True, rescale_learned_sigmas=True, timestep_respacing="")
        self.lib = _lib.lib()
        with torch.cuda.device(self.dev):
            self._bind_engine()
            z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=self.dev)
            # mixed-size mode: photos and outputs live in byte arenas, each document at a 16-byte aligned offset
            img = (docs, height, width, 3) if max_pixels is None else (3 * max_pixels + 16 * docs,)
            self.buf = {"y512": z(docs, 3, 512, 512), "mask_cat": z(docs, 1, 512, 512), "mask_y512": z(docs, 384, 64, 64),
                        "line_msk": z(docs, 64, 64, 64), "x_T": z(docs * n_batch, 2, 64, 64),
                        "photo_u8": z(*img, dt=torch.uint8)}
            self.init_flow0 = z(docs, 2, 64, 64)                       # evaluation.py:180 (use_init_flow=False)
            self.map64 = z(docs, 2, 64, 64)
            self.out_u8 = z(*img, dt=torch.uint8)
            self.out_host = torch.empty(img, dtype=torch.uint8).pin_memory()
            if max_pixels is not None:                                # run_device's unwarp table (host plan -> device copy)
                self._table = z(table_bytes(docs), dt=torch.uint8)
                self._table_host = torch.empty(table_bytes(docs), dtype=torch.uint8).pin_memory()
                self._ev_table = torch.cuda.Event()
        self.h2d_bytes = sum(v.numel() * v.element_size() for v in self.buf.values())
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

    # ---- device-resident inputs: dict with y512, mask_cat, mask_y512, line_msk, x_T, photo_u8 (all on self.dev)
    def _enqueue_sampling(self, d: dict):
        """static conditioning -> S-step DDIM loop -> hypothesis mean (map64), on the current stream."""
        self.eng.static_forward(d["y512"], d["mask_cat"], d["mask_y512"], d["line_msk"])
        self.eng.sample(d["x_T"], self.init_flow0, self.tables, self.t_scaled, self.a, self.b, None, self.map64)

    def _enqueue_unwarp(self, d: dict):
        """fused upsample + affine + bilinear unwarp of the full-resolution photo, on the current stream."""
        out = d.get("out_u8", self.out_u8)
        _lib.check(self.lib.dvd_unwarp_u8(_lib.ptr(d["photo_u8"]), _lib.ptr(self.map64), _lib.ptr(out), self.docs, 3,
                                          self.H, self.W, 64, 64, AFFINE, _lib.stream_ptr()), "dvd_unwarp_u8")

    def _enqueue_unwarp_mixed(self, d: dict):
        """mixed-size unwarp of the batch planned into the device table d["table"] (one launch whatever the composition)."""
        _lib.check(self.lib.dvd_unwarp_u8_mixed(_lib.ptr(d["table"]), 3, _lib.ptr(self.map64), _lib.stream_ptr()), "dvd_unwarp_u8_mixed")

    def _check_photos(self, photos, device: torch.device, lo: int) -> list:
        """Validates the photos of a mixed-size batch (lo..docs uint8 HWC RGB tensors on `device`, at most max_pixels in all)."""
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
        """one [H,W,3] view per photo, packed at 16-byte aligned offsets"""
        views, off = [], 0
        for p in photos:
            views.append(arena[off:off + p.numel()].view(p.shape))
            off = (off + p.numel() + 15) & ~15
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
        unwarp) and replayed (the library never allocates or synchronises, so every entry point is capturable).

        Mixed-size mode: d["photo_u8"] is a list of exactly `docs` uint8 HWC photos on the pipeline's device (read in place);
        returns a list of views into the device output arena, overwritten by the next call."""
        self._check_weights()
        if self.max_pixels is not None:
            return self._run_device_mixed(d)
        with torch.cuda.device(self.dev):
            self._run("sampling", d, self.SAMPLING_KEYS, self._enqueue_sampling)
            self._run("unwarp", d, ("photo_u8",), self._enqueue_unwarp)
        return self.out_u8

    def _run_device_mixed(self, d: dict) -> list:
        photos = self._check_photos(d["photo_u8"], self.dev, self.docs)
        with torch.cuda.device(self.dev):
            self._run("sampling", d, self.SAMPLING_KEYS, self._enqueue_sampling)
            outs = self._arena_views(self.out_u8, photos)
            self._ev_table.synchronize()                               # the previous upload has read the pinned table
            plan_mixed(self._table_host, photos, outs, 64, 64)
            self._table.copy_(self._table_host, non_blocking=True)
            self._ev_table.record()
            self._run("unwarp", {"table": self._table}, ("table",), self._enqueue_unwarp_mixed)
        return outs

    # ---- pinned-host inputs -> host uint8 image (H2D and D2H inside the call)
    def _make_slots(self):
        """Two sets of device input / output buffers + copy streams: the uploads of batch i+1 and the download of batch i run
        underneath the kernels of the batch in between (the kernels themselves stay on the caller's stream, one batch at a time)."""
        self._h2d = torch.cuda.Stream(device=self.dev)
        self._d2h = torch.cuda.Stream(device=self.dev)
        self._slots = []
        for _ in range(2):
            buf = {k: torch.empty_like(v) for k, v in self.buf.items()}
            buf["out_u8"] = torch.empty_like(self.out_u8)
            slot = {"buf": buf, "out_host": torch.empty_like(self.out_host).pin_memory(), "used": False,
                    "ev_in": torch.cuda.Event(), "ev_photo": torch.cuda.Event(), "ev_done": torch.cuda.Event(), "ev_out": torch.cuda.Event()}
            if self.max_pixels is not None:
                buf["table"] = torch.empty_like(self._table)
                slot.update(table_host=torch.empty_like(self._table_host).pin_memory(), ev_table=torch.cuda.Event(), views=None)
            self._slots.append(slot)
        self._submitted = 0

    def submit_host(self, h: dict) -> int:
        """Enqueue one batch (pinned host inputs) without waiting for it; returns a ticket for `wait`.  At most two batches may be
        outstanding (a ticket must be waited for before the second-next submit).  The photo is only needed by the last kernel, so
        its upload also runs underneath this batch's own sampling.

        Mixed-size mode: h["photo_u8"] is a list of 1..docs uint8 HWC host photos and the other inputs have that many documents
        (x_T that many times n_batch); document slots past the list keep their earlier inputs, are sampled and not unwarped."""
        self._check_weights()
        if self.max_pixels is not None:
            return self._submit_host_mixed(h)
        with torch.cuda.device(self.dev):
            if self._slots is None:
                self._make_slots()
            main = torch.cuda.current_stream()
            ticket = self._submitted
            self._submitted += 1
            s = self._slots[ticket % 2]
            with torch.cuda.stream(self._h2d):
                if s["used"]:
                    self._h2d.wait_event(s["ev_done"])             # the kernels of batch ticket-2 have read this slot's inputs
                for k in self.SAMPLING_KEYS:
                    s["buf"][k].copy_(h[k], non_blocking=True)
                s["ev_in"].record()
                s["buf"]["photo_u8"].copy_(h["photo_u8"], non_blocking=True)
                s["ev_photo"].record()
            main.wait_event(s["ev_in"])
            if s["used"]:
                main.wait_event(s["ev_out"])                       # the download of batch ticket-2 has read this slot's output
            self._run("sampling", s["buf"], self.SAMPLING_KEYS, self._enqueue_sampling)
            main.wait_event(s["ev_photo"])
            self._run("unwarp", s["buf"], ("photo_u8", "out_u8"), self._enqueue_unwarp)
            s["ev_done"].record(main)
            with torch.cuda.stream(self._d2h):
                self._d2h.wait_event(s["ev_done"])
                s["out_host"].copy_(s["buf"]["out_u8"], non_blocking=True)
                s["ev_out"].record()
            s["used"] = True
        return ticket

    def _submit_host_mixed(self, h: dict) -> int:
        photos = self._check_photos(h["photo_u8"], torch.device("cpu"), 1)
        n = len(photos)
        for k in self.SAMPLING_KEYS:
            want = (n * self.n_batch if k == "x_T" else n,) + tuple(self.buf[k].shape[1:])
            if tuple(h[k].shape) != want:
                raise ValueError(f"{k}: expected shape {want} for {n} photos, got {tuple(h[k].shape)}")
        with torch.cuda.device(self.dev):
            if self._slots is None:
                self._make_slots()
            main = torch.cuda.current_stream()
            ticket = self._submitted
            self._submitted += 1
            s = self._slots[ticket % 2]
            buf = s["buf"]
            photo_dev = self._arena_views(buf["photo_u8"], photos)
            out_dev = self._arena_views(buf["out_u8"], photos)
            with torch.cuda.stream(self._h2d):
                if s["used"]:
                    self._h2d.wait_event(s["ev_done"])             # the kernels of batch ticket-2 have read this slot's inputs
                for k in self.SAMPLING_KEYS:
                    buf[k][:h[k].shape[0]].copy_(h[k], non_blocking=True)
                s["ev_in"].record()
                for dst, src in zip(photo_dev, photos):
                    dst.copy_(src, non_blocking=True)
                s["ev_photo"].record()
            main.wait_event(s["ev_in"])
            if s["used"]:
                main.wait_event(s["ev_out"])                       # the download of batch ticket-2 has read this slot's output
            self._run("sampling", buf, self.SAMPLING_KEYS, self._enqueue_sampling)
            # the device only waits for batch ticket-2 through events; the HOST rewrites the pinned table now, so the upload of
            # ticket-2 must have read it (normally long done)
            s["ev_table"].synchronize()
            plan_mixed(s["table_host"], photo_dev, out_dev, 64, 64)
            buf["table"].copy_(s["table_host"], non_blocking=True)
            s["ev_table"].record(main)
            main.wait_event(s["ev_photo"])
            self._run("unwarp", buf, ("table",), self._enqueue_unwarp_mixed)
            s["ev_done"].record(main)
            end = out_dev[-1].data_ptr() - buf["out_u8"].data_ptr() + out_dev[-1].numel()
            with torch.cuda.stream(self._d2h):
                self._d2h.wait_event(s["ev_done"])
                s["out_host"][:end].copy_(buf["out_u8"][:end], non_blocking=True)
                s["ev_out"].record()
            s["views"] = self._arena_views(s["out_host"], photos)
            s["used"] = True
        return ticket

    def wait(self, ticket: int):
        """Block until the batch of `ticket` is on the host; the returned pinned tensor (mixed-size mode: list of views into a
        pinned arena) is reused by the second-next submit."""
        s = self._slots[ticket % 2]
        s["ev_out"].synchronize()
        return s["out_host"] if self.max_pixels is None else s["views"]

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
