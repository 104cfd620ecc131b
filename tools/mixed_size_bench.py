"""End-to-end throughput of photos of MIXED sizes through DewarpPipeline (host path: submit_host / wait, two batches outstanding).

64 synthetic documents cycle over eight photo sizes; bf16x3, S = 3, n_batch = 2.  Three arms in one process:
  (i)   docs=1 per document, one fixed-size pipeline per distinct size (what a user with mixed photos had to do before);
  (ii)  one mixed-size pipeline, docs=16, max_pixels = the largest 16-document window of the set;
  (iii) the fixed-size pipeline with docs=16 on 1500x2000 photos only (all documents the same size: the ceiling for (ii)).
Inputs are pinned host tensors; every H2D / D2H copy is inside the timed region.  MSB_PASSES sets the timed passes over the set."""
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import synth_workload as synth                                           # noqa: E402
from dvd_b200.model import DiT                                          # noqa: E402
from dvd_b200.pipeline import DewarpPipeline                            # noqa: E402

SIZES = [(1500, 2000), (2000, 1500), (4032, 3024), (3024, 4032), (1200, 1600), (1333, 999), (2448, 3264), (600, 450)]
KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")
N_DOCS, BATCH = 64, 16


def host_doc(i, H, W):
    d = synth.make_doc_inputs(i, H=H, W=W)
    h = {k: d[k].contiguous().pin_memory() for k in KEYS}
    h["photo"] = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous().pin_memory()
    return h


def run_pipelined(jobs):
    """jobs: list of (pipe, host dict); submit_host each, waiting for the previous one (two outstanding)"""
    pending = None
    for pipe, h in jobs:
        t = pipe.submit_host(h)
        if pending is not None:
            pending[0].wait(pending[1])
        pending = (pipe, t)
    pending[0].wait(pending[1])


def timed(jobs, passes):
    run_pipelined(jobs)                                                  # warm-up pass: graph captures, first-touch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(passes):
        run_pipelined(jobs)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    dev = torch.device("cuda:0")
    passes = int(os.environ.get("MSB_PASSES", "3"))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    print(f"GPU: {gpu}")
    model = DiT(precision="bf16x3")
    model.load_state_dict(synth.make_state_dict(1234, live_only=True), strict=False)
    model.to(dev).eval()
    per_size = [host_doc(k, H, W) for k, (H, W) in enumerate(SIZES)]        # document i uses the inputs of size i % 8
    docs = [per_size[i % len(SIZES)] for i in range(N_DOCS)]
    kw = dict(diffusion_steps=3, n_batch=2, precision="bf16x3")
    res = {}

    # (i) docs=1, one pipeline per size
    pipes = {hw: DewarpPipeline(model, docs=1, height=hw[0], width=hw[1], **kw) for hw in SIZES}
    jobs = []
    for d in docs:
        h = {k: d[k] for k in KEYS}
        h["photo_u8"] = d["photo"].unsqueeze(0)
        jobs.append((pipes[tuple(d["photo"].shape[:2])], h))
    res["(i) docs=1, one pipeline per size"] = timed(jobs, passes)
    del pipes, jobs
    torch.cuda.empty_cache()

    # (ii) mixed-size pipeline, docs=16
    P = max(sum(d["photo"].shape[0] * d["photo"].shape[1] for d in docs[b:b + BATCH]) for b in range(0, N_DOCS, BATCH))
    pipe = DewarpPipeline(model, docs=BATCH, max_pixels=P, **kw)
    jobs = []
    for b in range(0, N_DOCS, BATCH):
        ds = docs[b:b + BATCH]
        h = {k: torch.cat([d[k] for d in ds]).pin_memory() for k in KEYS}
        h["photo_u8"] = [d["photo"] for d in ds]
        jobs.append((pipe, h))
    res[f"(ii) mixed sizes, docs=16, max_pixels={P}"] = timed(jobs, passes)
    del pipe, jobs
    torch.cuda.empty_cache()

    # (iii) fixed-size docs=16, 1500x2000 only
    pipe = DewarpPipeline(model, docs=BATCH, height=1500, width=2000, **kw)
    d0 = per_size[0]
    h = {k: torch.cat([d0[k]] * BATCH).pin_memory() for k in KEYS}
    h["photo_u8"] = torch.stack([d0["photo"]] * BATCH).pin_memory()
    res["(iii) fixed 1500x2000, docs=16 (ceiling)"] = timed([(pipe, h)] * (N_DOCS // BATCH), passes)

    print(f"{N_DOCS} documents cycling over {len(SIZES)} sizes {SIZES}; bf16x3, S=3, n_batch=2; submit_host/wait with two batches "
          f"outstanding; {passes} timed passes after one warm-up pass")
    for name, sec in res.items():
        print(f"{name:55s} {N_DOCS * passes / sec:7.1f} docs/s  ({sec * 1e3 / (N_DOCS * passes):.2f} ms per document)")


if __name__ == "__main__":
    main()
