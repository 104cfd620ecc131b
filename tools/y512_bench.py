"""The denoiser's y512 computed from the photo on the GPU: kernel time of the y512 launch and end-to-end DewarpPipeline throughput.

Kernel alone (CUDA events around a CUDA graph of 20 launches, 5 replays, median; rotating buffer sets larger than the L2 so every
launch reads its photos from HBM, as DewarpPipeline.profile_kernels times the unwarp): 16 x 4032x3024 and 16 x 1500x2000.  "rows"
is the traffic bound: the bytes of the source rows some output row reads (every 32-byte sector of such a row is touched once the
column step exceeds about 10 bytes) plus the fp32 output written.

End to end: DewarpPipeline docs=16, bf16x3, S = 3, n_batch = 2, 4032x3024 photos, host path (submit_host / wait, two batches
outstanding, every H2D / D2H copy inside the timed region), three arms alternating in one process:
  supplied       y512 supplied, resized on the host once outside the timed loop (bench.py's convention);
  supplied+cv2   y512 supplied, cv2.resize(photo, (512, 512), INTER_LINEAR) / 255 of each photo inside the loop (what a caller pays);
  from_photo     DewarpPipeline(y512_from_photo=True): no y512 upload, one extra launch in the sampling graph.
YB_ROUNDS sets the rounds, YB_BATCHES the batches per timed run."""
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import synth_workload as synth                                           # noqa: E402
from dvd_b200.inputs import launch_y512, plan_y512, table_bytes         # noqa: E402
from dvd_b200.model import DiT                                          # noqa: E402
from dvd_b200.pipeline import DewarpPipeline                            # noqa: E402

B = 16
N_LAUNCH = 20


def graph_time_us(launch, nbuf):
    """median over 5 replays of a graph of N_LAUNCH launches (launch(i) uses buffer set i % nbuf), µs per launch"""
    for i in range(nbuf):
        launch(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(N_LAUNCH):
            launch(i)
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / N_LAUNCH)
    ts.sort()
    return ts[2], ts[0], ts[-1]


def rows_read(H, W):
    """bytes of the distinct source rows the 512 output rows read (OpenCV's row taps sy, sy+1 clamped to the photo)"""
    f = ((np.arange(512) + 0.5) * (1.0 / (512.0 / H)) - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    return len(np.unique(np.clip(np.concatenate([s, s + 1]), 0, H - 1))) * W * 3


def kernel_bench(dev):
    print(f"kernel alone: CUDA graph of {N_LAUNCH} launches, median of 5 replays (min-max); inputs rotate over buffer sets larger than "
          f"the L2")
    for H, W in ((4032, 3024), (1500, 2000)):
        photo = synth.make_photo(H, W, 11, "page")[0].permute(1, 2, 0).to(torch.uint8).contiguous()
        per = B * H * W * 3 + B * 3 * 512 * 512 * 4
        nbuf = max(2, (300 << 20) // per + 1)
        ins = [torch.stack([photo] * B).to(dev) for _ in range(nbuf)]
        outs = [torch.empty((B, 3, 512, 512), dtype=torch.float32, device=dev) for _ in range(nbuf)]
        tables = []
        for k in range(nbuf):
            th = torch.empty(table_bytes(B), dtype=torch.uint8).pin_memory()
            plan_y512(th, list(ins[k].unbind(0)))
            tables.append(th.to(dev))
        med, lo, hi = graph_time_us(lambda i: launch_y512(tables[i % nbuf], outs[i % nbuf]), nbuf)
        rd, wr = B * rows_read(H, W), B * 3 * 512 * 512 * 4
        print(f"y512, {B} x {H}x{W}: {med:7.1f} us ({lo:.1f}-{hi:.1f})  rows {(rd + wr) / (med * 1e-6) / 1e9:7.1f} GB/s "
              f"(source rows {rd / 1e6:6.1f} MB + write {wr / 1e6:5.1f} MB; whole photos {B * H * W * 3 / 1e6:6.1f} MB)")
        del ins, outs, tables
        torch.cuda.empty_cache()


def e2e_bench(dev):
    H, W = 4032, 3024
    rounds = int(os.environ.get("YB_ROUNDS", "3"))
    nb = int(os.environ.get("YB_BATCHES", "4"))
    model = DiT(precision="bf16x3")
    model.load_state_dict(synth.make_state_dict(1234, live_only=True), strict=False)
    model.to(dev).eval()
    d = synth.make_doc_inputs(0, H=H, W=W)
    keys = ("mask_cat", "mask_y512", "line_msk", "x_T")
    h = {k: torch.cat([d[k]] * B).contiguous().pin_memory() for k in keys}
    h["photo_u8"] = torch.stack([d["photo"][0].permute(1, 2, 0).to(torch.uint8)] * B).contiguous().pin_memory()
    photos_np = h["photo_u8"].numpy()

    def resize_into(y):
        for i in range(B):
            r = cv2.resize(photos_np[i], (512, 512), interpolation=cv2.INTER_LINEAR)
            y[i].copy_(torch.from_numpy(r).permute(2, 0, 1).float().div_(255))

    y_fixed = torch.empty((B, 3, 512, 512), dtype=torch.float32).pin_memory()
    resize_into(y_fixed)
    y_loop = [torch.empty_like(y_fixed).pin_memory() for _ in range(2)]      # one per outstanding batch

    def with_cv2(i):
        y = y_loop[i % 2]                                                # batch i-2, which read this buffer, has been waited for
        resize_into(y)
        return dict(h, y512=y)

    kw = dict(diffusion_steps=3, n_batch=2, docs=B, height=H, width=W, precision="bf16x3")
    arms = {"supplied": (DewarpPipeline(model, **kw), lambda i: dict(h, y512=y_fixed)),
            "supplied+cv2": (DewarpPipeline(model, **kw), with_cv2),
            "from_photo": (DewarpPipeline(model, y512_from_photo=True, **kw), lambda i: h)}

    def run(pipe, inputs):
        pending = None
        for i in range(nb):
            t = pipe.submit_host(inputs(i))
            if pending is not None:
                pipe.wait(pending)
            pending = t
        pipe.wait(pending)

    for pipe, inputs in arms.values():
        run(pipe, inputs)                                                # warm-up: graph captures, first touch
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
        resize_into(y_loop[0])
    host_ms = (time.perf_counter() - t0) / 5 * 1e3
    print(f"end to end: DewarpPipeline docs={B}, bf16x3, S=3, n_batch=2, {H}x{W} photos, submit_host/wait with two batches "
          f"outstanding, {nb} batches per run, {rounds} rounds alternating the arms; host resize + /255 of {B} photos: {host_ms:.1f} ms "
          f"({torch.get_num_threads()} torch threads, {cv2.getNumThreads()} cv2 threads)")
    for name, (pipe, _) in arms.items():
        v = res[name]
        print(f"{name:14s} h2d {pipe.h2d_bytes / 1e6:6.1f} MB/batch  docs/s " + " ".join(f"{x:6.1f}" for x in v) +
              f"   mean {sum(v) / len(v):6.1f}")


def main():
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True).stdout.strip()
    print(f"GPU: {' | '.join(gpu.splitlines())}")
    with torch.cuda.device(dev):
        if "--e2e-only" not in sys.argv:
            kernel_bench(dev)
        if "--kernel-only" not in sys.argv:
            e2e_bench(dev)


if __name__ == "__main__":
    main()
