"""JPEG decode on the GPU: time per decode phase and end-to-end DewarpPipeline throughput with JPEG input.

Decode alone: 16 x 4032x3024 files (a synthetic page, cv2 quality 90 and 95, 4:2:0 and 4:4:4) already in device memory.  The whole
decode is timed with CUDA events around each call, the L2 overwritten before each (so the compressed bytes come from HBM), median of
JB_REPS; the phases are the kernels' device times from torch.profiler in a separate run.  "in" is the compressed GB/s, "out" the
RGB GB/s written.

End to end: DewarpPipeline docs=16, bf16x3, S = 3, n_batch = 2, 4032x3024 photos, y512_from_photo=True, host path (submit_host /
wait, two batches outstanding, every copy inside the timed region), three arms alternating in one process:
  photo_u8       decoded photos supplied (decoded once outside the timed loop: today's convention);
  cv2 8 threads  cv2.imdecode of the 16 files inside the loop on 8 host threads, then photo_u8;
  jpeg           DewarpPipeline(max_jpeg_bytes=...): the files are uploaded and decoded at the head of the sampling graph.
JB_ROUNDS sets the rounds, JB_BATCHES the batches per timed run."""
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import synth_workload as synth                                           # noqa: E402
from dvd_b200.inputs import (jpeg_hw, jpeg_table_bytes, jpeg_workspace_bytes, launch_jpeg, pack_jpeg,   # noqa: E402
                             plan_jpeg)
from dvd_b200.model import DiT                                          # noqa: E402
from dvd_b200.pipeline import DewarpPipeline                            # noqa: E402

B = 16
SAMPLING = {"420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}


def encode(rgb, q, s):
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(rgb[..., ::-1]), [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                                                           SAMPLING[s]])
    assert ok
    return buf.tobytes()


def page(H, W, seed):
    return synth.make_photo(H, W, seed, "page")[0].permute(1, 2, 0).to(torch.uint8).contiguous().numpy()


def decode_bench(dev):
    reps = int(os.environ.get("JB_REPS", "7"))
    H, W = 3024, 4032
    photos = [page(H, W, 11 + i) for i in range(4)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    print(f"decode alone: {B} x {H}x{W} files in device memory; CUDA events around each decode, L2 overwritten before each, median of "
          f"{reps} (min-max); phases: kernel device time from torch.profiler, mean of {reps}")
    for q in (90, 95):
        for s in ("420", "444"):
            files = [encode(photos[i % 4], q, s) for i in range(B)]
            hw = jpeg_hw(files)
            total = sum((len(f) + 15) & ~15 for f in files)
            host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
            offsets = pack_jpeg(files, host)
            arena = host.to(dev)
            outs = [torch.empty((h, w, 3), dtype=torch.uint8, device=dev) for h, w in hw]
            ws = torch.empty(jpeg_workspace_bytes(B, B * H * W, total), dtype=torch.uint8, device=dev)
            th = torch.empty(jpeg_table_bytes(B), dtype=torch.uint8, pin_memory=True)
            plan_jpeg(files, th, ws.numel(), arena, offsets, outs)
            table = th.to(dev)
            launch_jpeg(table, ws)
            torch.cuda.synchronize()
            ref = cv2.imdecode(np.frombuffer(files[0], np.uint8), cv2.IMREAD_COLOR)[..., ::-1]
            assert np.array_equal(outs[0].cpu().numpy(), ref), "decode differs from cv2.imdecode"
            ts = []
            for i in range(reps):
                flush.fill_(i)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); launch_jpeg(table, ws); e1.record(); e1.synchronize()
                ts.append(e0.elapsed_time(e1))
            ts.sort()
            med = ts[len(ts) // 2]
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for i in range(reps):
                    flush.fill_(i)
                    launch_jpeg(table, ws)
                torch.cuda.synchronize()
            phases = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA and "k_jpeg" in ev.name:
                    name = ev.name.split("k_jpeg_")[1].split("(")[0]
                    phases[name] = phases.get(name, 0.0) + ev.device_time / reps / 1e3
            cin, cout = sum(map(len, files)), sum(h * w * 3 for h, w in hw)
            print(f"q{q} {s}: {cin / 1e6:6.1f} MB -> {cout / 1e6:6.1f} MB  decode {med:6.3f} ms ({ts[0]:.3f}-{ts[-1]:.3f})  "
                  f"in {cin / (med * 1e-3) / 1e9:5.2f} GB/s  out {cout / (med * 1e-3) / 1e9:6.1f} GB/s")
            print("    phases (ms): " + "  ".join(f"{k} {v:.3f}" for k, v in phases.items()))
            del arena, outs, ws
            torch.cuda.empty_cache()


def e2e_bench(dev):
    H, W = 4032, 3024
    rounds = int(os.environ.get("JB_ROUNDS", "3"))
    nb = int(os.environ.get("JB_BATCHES", "4"))
    model = DiT(precision="bf16x3")
    model.load_state_dict(synth.make_state_dict(1234, live_only=True), strict=False)
    model.to(dev).eval()
    d = synth.make_doc_inputs(0, H=H, W=W)
    keys = ("mask_cat", "mask_y512", "line_msk", "x_T")
    h = {k: torch.cat([d[k]] * B).contiguous().pin_memory() for k in keys}
    rgb = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous().numpy()
    files = [encode(rgb if i % 2 == 0 else np.ascontiguousarray(rgb[:, ::-1]), 90, "420") for i in range(B)]
    decoded = [np.ascontiguousarray(cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR)[..., ::-1]) for f in files]
    photo_fixed = torch.from_numpy(np.stack(decoded)).pin_memory()
    photo_loop = [torch.empty_like(photo_fixed).pin_memory() for _ in range(2)]      # one per outstanding batch
    pool = ThreadPoolExecutor(8)

    def decode_into(dst):
        def one(i):
            dst[i].copy_(torch.from_numpy(cv2.imdecode(np.frombuffer(files[i], np.uint8), cv2.IMREAD_COLOR)[..., ::-1].copy()))
        list(pool.map(one, range(B)))

    def with_cv2(i):
        p = photo_loop[i % 2]                                            # batch i-2, which read this buffer, has been waited for
        decode_into(p)
        return dict(h, photo_u8=p)

    kw = dict(diffusion_steps=3, n_batch=2, docs=B, height=H, width=W, precision="bf16x3", y512_from_photo=True)
    arms = {"photo_u8": (DewarpPipeline(model, **kw), lambda i: dict(h, photo_u8=photo_fixed)),
            "cv2 8 threads": (DewarpPipeline(model, **kw), with_cv2),
            "jpeg": (DewarpPipeline(model, max_jpeg_bytes=max(map(len, files)), **kw), lambda i: dict(h, photo_jpeg=files))}

    def run(pipe, inputs):
        pending = None
        for i in range(nb):
            t = pipe.submit_host(inputs(i))
            if pending is not None:
                pipe.wait(pending)
            pending = t
        return pipe.wait(pending)

    outs = {}
    for name, (pipe, inputs) in arms.items():
        outs[name] = run(pipe, inputs).clone()                           # warm-up: graph captures, first touch
    same = all(torch.equal(outs["photo_u8"], o) for o in outs.values())
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for name, (pipe, inputs) in arms.items():
            t0 = time.perf_counter()
            run(pipe, inputs)
            torch.cuda.synchronize()
            res[name].append(B * nb / (time.perf_counter() - t0))
    t0 = time.perf_counter()
    for _ in range(5):
        decode_into(photo_loop[0])
    host_ms = (time.perf_counter() - t0) / 5 * 1e3
    print(f"end to end: DewarpPipeline docs={B}, bf16x3, S=3, n_batch=2, y512_from_photo, {H}x{W} photos (cv2 q90 4:2:0, "
          f"{sum(map(len, files)) / B / 1e6:.2f} MB a file), submit_host/wait with two batches outstanding, {nb} batches per run, "
          f"{rounds} rounds alternating the arms; cv2.imdecode of {B} files on 8 threads: {host_ms:.1f} ms; pages of the three arms "
          f"byte-identical: {same}")
    for name, (pipe, _) in arms.items():
        v = res[name]
        print(f"{name:14s} h2d {pipe.h2d_bytes / 1e6:6.1f} MB/batch  docs/s " + " ".join(f"{x:6.1f}" for x in v) +
              f"   mean {sum(v) / len(v):6.1f}  ({min(v):.1f}-{max(v):.1f})")


def main():
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
    print(f"GPU: {' | '.join(gpu.splitlines())}")
    with torch.cuda.device(dev):
        if "--e2e-only" not in sys.argv:
            decode_bench(dev)
        if "--decode-only" not in sys.argv:
            e2e_bench(dev)


if __name__ == "__main__":
    main()
