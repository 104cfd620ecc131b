#!/usr/bin/env python
"""bench.py — dewarped docs/sec (DDIM sampling + unwarp) on N B200s, one process per GPU.

    python bench.py --gpus 1 --steps 10 --warmup 3                  # our arm, N=1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W    # N>1 (document-sharded, no collective)
    python bench.py --impl reference ...                             # the UNMODIFIED reference on the host CPU (baseline/_ref)

One "step" = one batch of `--docs` synthetic documents per GPU through the whole hot path:
static conditioning (pyramid, embeds) -> S-step DDIM sampling (n_batch hypotheses) -> hypothesis
mean -> fused upsample + bilinear unwarp of the H x W photo.  Workload at N=1 = BASELINE.json
configs[1] (val_TDiff batch 1, 2000x1500 photo, S=3, n_batch=2).
  value : docs/s with the inputs already resident in HBM
  e2e   : the same through the public API with pinned-host inputs (H2D inside the timed region)
          and the unwarped uint8 image read back to the host (D2H inside the timed region)
Precision: the timed mode is `bf16x3` (tensor cores, split-precision operands, fp32-accurate: the mode that meets every
accuracy gate); the single-pass `bf16` mode and the FFMA `fp32` mode are measured beside it (N=1) as `bf16_mode` / `fp32_mode`.
Baselines reported beside the number (rank 0, N=1, after the timed region): `cpu_baseline` (one document through the reference
on the host cores, which also yields the `parity` object: our output against the reference's on the same document),
`torch_b200` (the reference's own modules on this GPU, TF32 off / on) and `preprocessing_ms` (the reference's three
preprocessing networks on this GPU, timed separately as north_star asks).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DVD_PRECISION", "bf16x3"), choices=["bf16x3", "bf16", "fp32"])
    ap.add_argument("--docs", type=int, default=1, help="documents per step per GPU")
    ap.add_argument("--total-docs", type=int, default=0, help="strong scaling: this many documents per step over ALL GPUs (BASELINE configs[2])")
    ap.add_argument("--height", type=int, default=1500)
    ap.add_argument("--width", type=int, default=2000)
    ap.add_argument("--diffusion-steps", type=int, default=3)
    ap.add_argument("--n-batch", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip bf16_mode / fp32_mode / torch_b200 / preprocessing / drop-in API legs")
    ap.add_argument("--save-doc0", default="", help="(reference arm) also write the map and the uint8 image of document 0 to this .npz")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="(our arm, rank 0) after the timed steps, write what the last timed step computed as DIR/<name>.npy in float32: "
                         "image (the dewarped photo that run_device returns, or a fixed seeded sample of it past 64 MiB in all) and "
                         "map64 (the sampled backward map it was unwarped with: an intermediate result, kept for finer comparison)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


def workload_name(a):
    return (f"val_TDiff batch {a.docs}/GPU: S={a.diffusion_steps} DDIM steps x n_batch={a.n_batch} hypotheses + unwarp of a "
            f"{a.width}x{a.height} (WxH) synthetic photo")


def config_dict(a):
    """Identical for both arms (the driver compares them)."""
    return {"workload": workload_name(a), "docs_per_step_per_gpu": a.docs, "photo_hw": [a.height, a.width],
            "diffusion_steps": a.diffusion_steps, "n_batch": a.n_batch, "weights": "random-init (synth_workload.py seed 1234)",
            "l2": "GPU arm: 256 MiB flush write between timed iterations (value, synchronous e2e); pipelined e2e and the CPU arm stream a new "
                  "document every step"}


# ------------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1])); mx.append(float(p[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            hi = [s for s in sm if s >= 0.5 * max(sm)] or sm          # samples under load
            out = {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def algorithmic_gflop_per_doc(S, n_batch):
    """SURVEY.md §8(d): live, hoisted FLOPs only."""
    return 101.87 + n_batch * S * 262.52


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each array as out_dir/<name>.npy in float32, smallest first, whole while it fits in what is left of DUMP_BYTES.  An
    array that does not fit is written as a 1-D sample at fixed positions (seeded, sorted, identical from run to run), so that two
    builds of the project can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES // 4 - 1024 * len(arrays)                          # float32 elements, minus room for the .npy headers
    for name, t in sorted(arrays.items(), key=lambda kv: kv[1].numel()):
        x = t.detach().float().cpu()
        if x.numel() > left:
            idx = torch.randperm(x.numel(), generator=torch.Generator().manual_seed(0))[:left].sort().values
            x = x.flatten()[idx]
        left -= x.numel()
        np.save(os.path.join(out_dir, name + ".npy"), x.numpy())


def psnr_db(a: torch.Tensor, b: torch.Tensor) -> float:
    mse = float(((a.double() - b.double()) ** 2).mean())
    return 99.0 if mse == 0 else 10 * math.log10(255.0 ** 2 / mse)


# ------------------------------------------------------------------------------------------------ reference legs (host CPU / stock torch)
class ReferenceRunner:
    """One whole document per call through the reference's own implementation of the path, as written (12 DiT blocks, nothing
    hoisted, its debug PNG dumps): evaluation.py:80-138 + :300-306 + visualization_utils.py:75-77.
    kind = "reference": the UNMODIFIED reference imported from baseline/_ref (or /root/reference) through oracle/ref_shims;
    kind = "port": the oracle's restatement, only when the reference tree is absent."""

    def __init__(self, a, device="cpu"):
        import synth_workload as synth
        self.a, self.synth, self.device = a, synth, device
        self.sd = synth.make_state_dict(1234)
        self.kind = "port"
        try:
            from oracle import ref_harness as RH
            if RH.available():
                self.RH = RH
                self.model = RH.build_reference_model(self.sd).to(device)
                self.kind = "reference"
        except Exception as e:                                   # noqa: BLE001 - fall back to the port, say why
            self.why = repr(e)[:200]

    def doc(self, doc_id: int):
        """-> (uint8 HWC image, map64 [1,2,64,64] on the CPU, seconds)."""
        a = self.a
        inp = self.synth.make_doc_inputs(doc_id, H=a.height, W=a.width)
        photo = inp.pop("photo")
        t0 = time.perf_counter()
        with torch.no_grad():
            if self.kind == "reference":
                dev = torch.device(self.device)
                inp_d = {k: v.to(dev) for k, v in inp.items()}
                sample, _ = self.RH.reference_sample(self.model, inp_d, S=a.diffusion_steps, n_batch=a.n_batch, seed=2000 + doc_id)
                _, img = self.RH.reference_unwarp(sample, photo.to(dev))
                out = img[0].permute(1, 2, 0).cpu().numpy().astype("uint8")
                m = sample.cpu()
            else:
                from oracle import dvd_oracle as O
                m = O.sample(self.sd, inp, S=a.diffusion_steps, n_batch=a.n_batch, as_written=True)
                out = O.to_uint8_hwc(O.unwarp(m, photo))
        if self.device != "cpu":
            torch.cuda.synchronize()
        return out, m, time.perf_counter() - t0


def run_reference(a):
    """--impl reference: K whole documents (after W warm-up documents) through the reference on ALL host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the reference places its constant tensors on dist_util.dev() (= cuda when one is visible): hide the GPUs so that the CPU arm
    # really is the reference's CPU path (this process has not touched CUDA yet)
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    torch.set_num_threads(os.cpu_count())
    r = ReferenceRunner(a)
    if a.save_doc0:
        import numpy as np
        img, m, _ = r.doc(0)
        np.savez(a.save_doc0, img=img, map=m.numpy())
    for i in range(a.warmup):
        r.doc(i)
    ts = [r.doc(a.warmup + i)[2] for i in range(a.steps)]
    sec = sum(ts) / len(ts)
    value = a.docs / sec
    line = {"impl": "reference", "metric": "dewarped docs/sec (sampling+unwarp)", "value": value, "unit": "docs/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(a),
            "p50_latency_ms": statistics.median(ts) * 1e3,
            "cpu_baseline": {"value": value, "unit": "docs/s", "cores": torch.get_num_threads(), "kind": r.kind,
                             "sample": "every step = ONE WHOLE document through the reference as written (S x n_batch denoiser forwards with all 12 "
                                       "DiT blocks, its debug PNG dumps, full-size upsample + grid_sample + uint8 cast); no extrapolation"},
            "e2e": {"value": value, "unit": "docs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def torch_b200_leg(a, dev):
    """The reference's own modules on this GPU (stock cuDNN / cuBLAS kernels), as run_sampling.py would run them
    (cudnn.benchmark=True, run_sampling.py:27): whole documents, TF32 off and on.  The >= 10x target's denominator."""
    out = {}
    try:
        torch.backends.cudnn.benchmark = True
        r = ReferenceRunner(a, device=str(dev))
        if r.kind != "reference":
            return {"unavailable": "reference tree (baseline/_ref) not present"}
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            r.doc(0); r.doc(1)
            ts = [r.doc(2 + i)[2] for i in range(3)]
            out[name + "_docs_per_s"] = 1.0 / (sum(ts) / len(ts))
        out["what"] = "UNMODIFIED reference modules (baseline/_ref) on cuda: whole documents as written, wall clock with synchronize, 3 timed after 2 warm-up"
    except Exception as e:                                       # noqa: BLE001
        out["error"] = repr(e)[:300]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = True
    return out


def preprocessing_leg(dev):
    """north_star: the segmentation / line preprocessing models stay the reference modules and are timed separately.
    Random-init reference modules (val_TDiff.py:58-74) on a 288 x 288 input, CUDA events, ms per document."""
    out = {}
    try:
        from oracle import ref_harness as RH
        if not RH.available():
            return {"unavailable": "reference tree (baseline/_ref) not present"}
        nets = RH.build_preprocessing_nets()
        x = torch.rand(1, 3, 288, 288, device=dev)
        with torch.no_grad():
            for name, m in nets.items():
                m = m.to(dev)
                try:
                    for _ in range(3):
                        m(x)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(5):
                        m(x)
                    e1.record(); e1.synchronize()
                    out[name] = e0.elapsed_time(e1) / 5
                except Exception as e:                           # noqa: BLE001
                    out[name] = "error: " + repr(e)[:120]
        out["what"] = ("reference modules, random-init, batch 1 @288x288, fp32 stock kernels; GeoTr_Seg_Inf = U2NETP + GeoTr whose GeoTr half is "
                       "dead when use_init_flow=False (evaluation.py:176-180)")
    except Exception as e:                                       # noqa: BLE001
        out["error"] = repr(e)[:300]
    return out


def dropin_api_leg(a, model, dev, n_docs=12):
    """The drop-in path a user of run_sampling.py runs: dvd_b200.evaluation.run_evaluation_docunet (evaluation.py:142-327 replacement) over
    a loader of synthetic documents, one document per call like the reference, with stand-in preprocessing nets that return prepared
    device tensors (the real ones are timed separately in `preprocessing_ms`).  Wall clock over the whole loop, docs/s."""
    import synth_workload as synth
    from dvd_b200.evaluation import run_evaluation_docunet
    from dvd_b200.sampler import create_gaussian_diffusion
    out = {"api": "dvd_b200.evaluation.run_evaluation_docunet (drop-in for train_settings/dvd/evaluation.py:142-327), 1 document per call"}
    try:
        docs = [synth.make_doc_inputs(500 + i, H=a.height, W=a.width) for i in range(3)]
        dd = [{k: v.to(dev) for k, v in d.items() if k != "photo"} for d in docs]
        state = {"i": 0}

        class Env:
            train_mode = "stage_1_dit_cross"; iter = True; use_gt_mask = False; use_line_mask = True; use_init_flow = False
            clip_denoised = False; n_batch = a.n_batch; time_variant = True; visualize = True; eval_dataset_name = "bench"

        class Settings:
            env = Env(); name = "dropin"

        class Dewarp(torch.nn.Module):
            def forward(self, x):
                return None, dd[state["i"] % 3]["mask_cat"]

        class Seg(torch.nn.Module):
            def forward(self, x):
                parts = dd[state["i"] % 3]["mask_y512"].split(64, dim=1)
                return (x, None) + tuple(parts)

        class Line(torch.nn.Module):
            def forward(self, x):
                v = dd[state["i"] % 3]["line_msk"]
                state["i"] += 1
                return v, None

        loader = [{"source_image": docs[i % 3]["y512"], "source_image_ori": docs[i % 3]["photo"], "path": [f"/data/doc{i}.png"]}
                  for i in range(n_docs)]
        diffusion = create_gaussian_diffusion(steps=a.diffusion_steps, noise_schedule="cosine", predict_xstart=True, rescale_timesteps=True,
                                              rescale_learned_sigmas=True, timestep_respacing="")
        import contextlib, io
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as td, contextlib.redirect_stdout(io.StringIO()):     # the driver prints "Elapsed time ..." like the reference
            os.chdir(td)
            try:
                for vis, key in ((False, "docs_per_s_sampling_only"), (True, "docs_per_s_with_unwarp_and_png")):
                    Env.visualize = vis
                    state["i"] = 0
                    run_evaluation_docunet(Settings, None, loader[:3], diffusion, model, Dewarp(), Line(), Seg())      # warm-up (graph capture)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    run_evaluation_docunet(Settings, None, loader, diffusion, model, Dewarp(), Line(), Seg())
                    torch.cuda.synchronize()
                    out[key] = n_docs / (time.perf_counter() - t0)
            finally:
                os.chdir(cwd)
        out["note"] = ("per call: F.interpolate of the 512x512 photo, the stand-in nets, six device copies + ONE CUDA-graph replay of the whole "
                       "sampling, uint8 photo upload, fused unwarp, D2H, PNG encode on worker threads")
    except Exception as e:                                       # noqa: BLE001
        out["error"] = repr(e)[:300]
    return out


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(a):
    import torch.distributed as dist
    import synth_workload as synth                          # synthetic workload generator (no oracle code on this arm)
    import dvd_b200                                          # noqa: F401
    from dvd_b200 import _lib
    from dvd_b200.model import DiT
    from dvd_b200.pipeline import DewarpPipeline

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()
    scaling = "weak"
    if a.total_docs:                                        # strong scaling: a fixed batch of documents split over the ranks
        assert a.total_docs % world == 0, "--total-docs must be divisible by the number of GPUs"
        a.docs = a.total_docs // world
        scaling = "strong"

    # ---- synthetic workload: documents sharded by rank (doc id = step*world*docs + rank*docs + j); no collective on the path
    sd = synth.make_state_dict(1234, live_only=True)
    model = DiT(precision=a.precision)
    model.load_state_dict(sd, strict=False)
    model.to(dev)
    n_var = 2                                               # distinct input sets that the steps rotate through
    host_sets = []
    for v in range(n_var):
        docs = [synth.make_doc_inputs(1000 * rank + v * a.docs + j, H=a.height, W=a.width) for j in range(a.docs)]
        hs = {k: torch.cat([d[k] for d in docs]).contiguous().pin_memory() for k in ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")}
        hs["photo_u8"] = torch.cat([d["photo"] for d in docs]).permute(0, 2, 3, 1).to(torch.uint8).contiguous().pin_memory()
        host_sets.append(hs)
    dev_sets = [{k: v.to(dev) for k, v in hs.items()} for hs in host_sets]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(precision, steps, warmup, with_e2e=True, keep_last=False):
        pipe = DewarpPipeline(model, diffusion_steps=a.diffusion_steps, n_batch=a.n_batch, docs=a.docs, height=a.height, width=a.width,
                              precision=precision)

        def timed(fn):
            for i in range(warmup):
                fn(i)
            barrier()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            pipe.kernel_launches = 0
            for i in range(steps):
                flush.fill_(i & 0xFF)                                         # L2 flush between timed iterations (not timed)
                evs[i][0].record()
                fn(warmup + i)
                evs[i][1].record()
            barrier()
            return [s.elapsed_time(e) for s, e in evs], pipe.kernel_launches

        def timed_e2e_pipelined():
            """Throughput form of the same API (submit_host / wait, two batches outstanding): the uploads of batch i+1 and the download
            of batch i overlap the kernels in between.  Every batch's H2D and D2H copies are inside the timed region."""
            pending = None
            for i in range(warmup):
                t = pipe.submit_host(host_sets[i % n_var])
                if pending is not None:
                    pipe.wait(pending)
                pending = t
            pipe.wait(pending); pending = None
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                t = pipe.submit_host(host_sets[(warmup + i) % n_var])
                if pending is not None:
                    pipe.wait(pending)
                pending = t
            pipe.wait(pending)                                                # the last image is on the host
            e1.record()
            barrier()
            return e0.elapsed_time(e1)

        ms_dev, launches = timed(lambda i: pipe.run_device(dev_sets[i % n_var]))           # (1) device-resident inputs
        res = {"pipe": pipe, "ms_dev": ms_dev, "launches": launches}
        if keep_last:                                                      # the e2e legs below overwrite pipe.map64
            res["last"] = {"map64": pipe.map64.clone(), "image": pipe.out_u8.clone()}
        if with_e2e:
            res["ms_e2e"], _ = timed(lambda i: pipe.run_host(host_sets[i % n_var]))        # (2) synchronous public-API calls: latency
            res["ms_e2e_pipe"] = timed_e2e_pipelined()                                     # (3) two batches outstanding: throughput
        return res

    def reduce_max(vals):
        if world == 1:
            return vals
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                              # max over ranks (timing only; not on the data path)
        return [float(x) for x in t]

    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.05)
    main = measure(a.precision, a.steps, a.warmup, keep_last=bool(a.dump_outputs) and rank == 0)
    clocks = sampler.stop() if sampler else None
    if "last" in main:
        dump_outputs(a.dump_outputs, main.pop("last"))
    pipe = main["pipe"]
    tot_dev, tot_e2e = reduce_max([sum(main["ms_dev"]) / 1e3, min(sum(main["ms_e2e"]), main["ms_e2e_pipe"]) / 1e3])
    docs_total = a.docs * a.steps * world
    value, e2e = docs_total / tot_dev, docs_total / tot_e2e

    if rank == 0:
        peaks, which = measured_peaks()
        prof = pipe.profile_kernels(dev_sets[0])                             # CUDA-event timing of the dominant kernels, L2-flushed
        gflop = algorithmic_gflop_per_doc(a.diffusion_steps, a.n_batch) * a.docs
        dtype = {"bf16x3": "bf16x3 (split 16-bit operand pairs, 3 tcgen05 passes per k-step - 2 in the decoder q|k|v GEMMs and the pyramid convs -, fp32 accumulate: fp32-accurate)", "bf16": "bf16", "fp32": "f32"}[a.precision]
        line = {"metric": "dewarped docs/sec (sampling+unwarp)", "value": value, "unit": "docs/s", "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": tot_dev / a.steps * 1e3, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config_dict(a),
                "run": {"cuda_graph": pipe.use_graph, "parallelism": f"document-sharded x{world}, no collective", "precision": a.precision},
                "p50_latency_ms": statistics.median(main["ms_dev"]),
                "e2e": {"value": e2e, "unit": "docs/s", "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
                        "p50_latency_ms": statistics.median(main["ms_e2e"]), "io": "uint8 HWC photo in, uint8 HWC dewarped image out",
                        "mode": "submit_host/wait, two batches outstanding (uploads and downloads overlap the kernels of the batch in between)",
                        "synchronous_docs_per_s": a.docs * a.steps * world / (sum(main["ms_e2e"]) / 1e3)},      # rank 0's clock x world
                "gpu_launches": int(main["launches"]),
                "clocks": clocks,
                "denoiser_tflops_effective": gflop / 1e3 / (tot_dev / a.steps / 1.0) if tot_dev > 0 else None,
                "roofline": prof["roofline"], "roofline_unwarp": prof["roofline_unwarp"], "kernel_share": prof.get("share"),
                "peaks": which}
        extras = world == 1 and not a.no_extras
        if extras:
            # ---- the other two precision modes on the same workload (device-resident value + pipelined e2e)
            try:
                for prec, key, st in (("bf16", "bf16_mode", a.steps), ("fp32", "fp32_mode", min(a.steps, 3))):
                    if prec == a.precision:
                        continue
                    r = measure(prec, st, 3, with_e2e=(prec == "bf16"))
                    o = {"value": a.docs * st / (sum(r["ms_dev"]) / 1e3), "unit": "docs/s", "ms_per_step": sum(r["ms_dev"]) / st,
                         "gpu_launches": int(r["launches"])}
                    if prec == "bf16":
                        o["e2e"] = a.docs * st / (min(sum(r["ms_e2e"]), r["ms_e2e_pipe"]) / 1e3)
                        pr = r["pipe"].profile_kernels(dev_sets[0], iters=4, with_unwarp=False)
                        o["roofline_frac"] = pr["roofline"]["frac"]; o["gemm_tflops"] = pr["roofline"]["achieved"]
                        o["attention_tflops"] = pr["roofline"]["attention_tflops"]
                        o["accuracy"] = "single pass: map error ~6e-4 normalised (0.6 px at 2000 px), image PSNR below the 45 dB gate - reduced-accuracy mode"
                    else:
                        o["accuracy"] = "FFMA reference mode (no tensor cores), bit-reproducible"
                    line[key] = o
                    del r
            except Exception as e:                                           # noqa: BLE001
                line["bf16_mode_error"] = repr(e)[:300]
        if world == 1 and not a.no_cpu_baseline:
            # ---- one document through the reference on the host cores: the cpu_baseline AND the parity check of the timed precision
            # (a child process with the GPUs hidden: the reference follows torch.cuda.is_available() for its constant tensors)
            import numpy as np
            with tempfile.TemporaryDirectory() as td:
                f = os.path.join(td, "doc0.npz")
                cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0", "--save-doc0", f,
                       "--height", str(a.height), "--width", str(a.width), "--diffusion-steps", str(a.diffusion_steps), "--n-batch", str(a.n_batch)]
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
                if out.returncode != 0:
                    raise RuntimeError("cpu_baseline leg failed: " + out.stderr[-1500:])
                rl = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
                z = np.load(f)
                ref_img, ref_map = z["img"], torch.from_numpy(z["map"])
            sec = rl["ms_per_step"] / 1e3
            kind = rl["cpu_baseline"]["kind"]
            line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "docs/s", "cores": rl["cpu_baseline"]["cores"], "kind": kind,
                                    "sample": f"1 whole document through the reference as written ({sec:.1f} s: S x n_batch forwards with all 12 DiT "
                                              "blocks, debug PNG dumps, full-size unwarp + uint8 cast)"}

            class r:                                                          # noqa: N801 - just carries the label below
                pass
            r.kind = kind
            try:
                d0 = synth.make_doc_inputs(0, H=a.height, W=a.width)
                one = DewarpPipeline(model, diffusion_steps=a.diffusion_steps, n_batch=a.n_batch, docs=1, height=a.height, width=a.width,
                                     precision=a.precision)
                dset = {k: d0[k].to(dev).contiguous() for k in ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")}
                dset["photo_u8"] = d0["photo"].permute(0, 2, 3, 1).to(torch.uint8).contiguous().to(dev)
                img = one.run_device(dset).cpu()
                err = (one.map64.cpu() - ref_map).abs()
                line["parity"] = {"vs": f"{r.kind} on this box's CPU, document 0, same weights and seeded noise", "precision": a.precision,
                                  "map_err_mean_px_at_4032": float(err.mean()) * 2015.5, "map_err_max_px_at_4032": float(err.max()) * 2015.5,
                                  "map_err_mean_norm": float(err.mean()), "map_err_max_norm": float(err.max()),
                                  "image_psnr_db_uint8": psnr_db(img[0].float(), torch.from_numpy(ref_img).float()),
                                  "gates": "map <= 0.05 px mean / 0.5 px max; image PSNR >= 45 dB"}
            except Exception as e:                                           # noqa: BLE001
                line["parity_error"] = repr(e)[:300]
        if extras:
            line["torch_b200"] = torch_b200_leg(a, dev)
            if "fp32_docs_per_s" in line["torch_b200"]:
                line["torch_b200"]["speedup_vs_fp32"] = value / line["torch_b200"]["fp32_docs_per_s"]
                line["torch_b200"]["speedup_vs_tf32"] = value / line["torch_b200"]["tf32_docs_per_s"]
            line["preprocessing_ms"] = preprocessing_leg(dev)
            line["dropin_api"] = dropin_api_leg(a, model, dev)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
