"""Dewarping to a requested output size: kernel time of the sized uint8 launch and end-to-end DewarpPipeline throughput.

Kernel alone (CUDA events around a CUDA graph of 20 launches, 5 replays, median; rotating buffer sets larger than the L2 so every
launch reads its photos from HBM; smooth synthetic map, as in DewarpPipeline.profile_kernels):
  (a) dvd_unwarp_u8, 16 x 4032x3024 at full size (the baseline);
  (b) dvd_unwarp_u8_sized, same photos, long side 2048 (auto s = 2);
  (c) long side 1024 (auto s = 4);
  (d) long side 512 (auto s = 8);
  (e) as (c) on a mixed batch: 16 documents cycling over the eight sizes of tools/mixed_size_bench.py.
GB/s is compulsory traffic: photo bytes read + output bytes written, over the kernel time.

End to end: DewarpPipeline docs=16, bf16x3, S = 3, n_batch = 2, 4032x3024 photos, host path (submit_host / wait, two batches
outstanding, every H2D / D2H copy inside the timed region); out_size None vs long side 2048 vs long side 1024, the arms alternating
in one process.  RB_ROUNDS sets the rounds, RB_BATCHES the batches per timed run."""
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import synth_workload as synth                                           # noqa: E402
from dvd_b200 import _lib                                               # noqa: E402
from dvd_b200.model import DiT                                          # noqa: E402
from dvd_b200.pipeline import DewarpPipeline                            # noqa: E402
from dvd_b200.unwarp import AFFINE, plan_sized, sized_table_bytes       # noqa: E402

H, W, B = 4032, 3024, 16
MIXED = [(1500, 2000), (2000, 1500), (4032, 3024), (3024, 4032), (1200, 1600), (1333, 999), (2448, 3264), (600, 450)]
KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")
N_LAUNCH = 20


def long_side(n):
    """out_size callable: long side n, aspect kept"""
    return lambda h, w: (max(1, round(h * n / max(h, w))), max(1, round(w * n / max(h, w))))


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


def kernel_bench(dev):
    lib = _lib.lib()
    gen = torch.Generator(device="cpu").manual_seed(3005)
    smooth = torch.nn.functional.interpolate(torch.randn((1, 2, 8, 8), generator=gen) * 0.02, size=(64, 64), mode="bicubic",
                                             align_corners=True).clamp(-1, 1).repeat(B, 1, 1, 1).contiguous().to(dev)
    photo = synth.make_photo(H, W, 11, "page")[0].permute(1, 2, 0).to(torch.uint8).contiguous()
    per = B * H * W * 3
    nbuf = max(2, (300 << 20) // per + 1)
    ins = [torch.stack([photo] * B).to(dev) for _ in range(nbuf)]
    rows = []

    outs = [torch.empty_like(x) for x in ins]
    t = graph_time_us(lambda i: _lib.check(lib.dvd_unwarp_u8(_lib.ptr(ins[i % nbuf]), _lib.ptr(smooth), _lib.ptr(outs[i % nbuf]), B, 3,
                                                             H, W, 64, 64, AFFINE, _lib.stream_ptr()), "dvd_unwarp_u8"), nbuf)
    rows.append(("(a) dvd_unwarp_u8, full size", f"{B} x {H}x{W} -> {H}x{W}", "-", per, per, t))
    del outs

    def sized(name, photos_sets, out_shapes):
        """photos_sets[k]: list of device photos of buffer set k; out_shapes: per document (Ho, Wo)"""
        n = len(photos_sets)
        outs = [[torch.empty(s + (3,), dtype=torch.uint8, device=dev) for s in out_shapes] for _ in range(n)]
        tables, chosen = [], None
        for k in range(n):
            th = torch.empty(sized_table_bytes(len(out_shapes)), dtype=torch.uint8).pin_memory()
            _, chosen = plan_sized(th, photos_sets[k], outs[k], 64, 64, 0)
            tables.append(th.to(dev))
        rd = sum(p.numel() for p in photos_sets[0])
        wr = sum(o.numel() for o in outs[0])
        t = graph_time_us(lambda i: _lib.check(lib.dvd_unwarp_u8_sized(_lib.ptr(tables[i % n]), 3, _lib.ptr(smooth), _lib.stream_ptr()),
                                               "dvd_unwarp_u8_sized"), n)
        return rd, wr, t, sorted(set(chosen))

    for tag, n in (("(b)", 2048), ("(c)", 1024), ("(d)", 512)):
        shape = long_side(n)(H, W)
        rd, wr, t, ss = sized(tag, [list(x.unbind(0)) for x in ins], [shape] * B)
        rows.append((f"{tag} sized, long side {n}", f"{B} x {H}x{W} -> {shape[0]}x{shape[1]}", ss, rd, wr, t))
    del ins
    torch.cuda.empty_cache()

    mixed = [MIXED[i % len(MIXED)] for i in range(B)]
    mphotos = [synth.make_photo(h, w, 20 + k, "page")[0].permute(1, 2, 0).to(torch.uint8).contiguous() for k, (h, w) in enumerate(MIXED)]
    mper = sum(h * w * 3 for h, w in mixed)
    mbuf = max(2, (300 << 20) // (mper + sum(long_side(1024)(h, w)[0] * long_side(1024)(h, w)[1] * 3 for h, w in mixed)) + 1)
    sets = [[mphotos[i % len(MIXED)].to(dev) for i in range(B)] for _ in range(mbuf)]
    rd, wr, t, ss = sized("(e)", sets, [long_side(1024)(h, w) for h, w in mixed])
    rows.append(("(e) sized, long side 1024, mixed batch", f"{B} docs over {len(MIXED)} sizes", ss, rd, wr, t))

    print(f"kernel alone: CUDA graph of {N_LAUNCH} launches, median of 5 replays (min-max); inputs rotate over buffer sets larger than "
          f"the L2; smooth synthetic map (amplitude 0.02)")
    base = rows[0][5][0]
    for name, what, ss, rd, wr, (med, lo, hi) in rows:
        print(f"{name:42s} {what:34s} s={str(ss):8s} {med:8.1f} us ({lo:.1f}-{hi:.1f})  {(rd + wr) / (med * 1e-6) / 1e9:7.1f} GB/s "
              f"(read {rd / 1e6:6.1f} MB + write {wr / 1e6:6.1f} MB)  {med / base:5.2f}x (a)")


def e2e_bench(dev):
    rounds = int(os.environ.get("RB_ROUNDS", "3"))
    nb = int(os.environ.get("RB_BATCHES", "4"))
    model = DiT(precision="bf16x3")
    model.load_state_dict(synth.make_state_dict(1234, live_only=True), strict=False)
    model.to(dev).eval()
    d = synth.make_doc_inputs(0, H=H, W=W)
    h = {k: torch.cat([d[k]] * B).contiguous().pin_memory() for k in KEYS}
    h["photo_u8"] = torch.stack([d["photo"][0].permute(1, 2, 0).to(torch.uint8)] * B).contiguous().pin_memory()
    kw = dict(diffusion_steps=3, n_batch=2, docs=B, height=H, width=W, precision="bf16x3")
    arms = {"out_size=None (4032x3024)": DewarpPipeline(model, **kw),
            "long side 2048": DewarpPipeline(model, out_size=long_side(2048), **kw),
            "long side 1024": DewarpPipeline(model, out_size=long_side(1024), **kw)}

    def run(pipe):
        pending = None
        for _ in range(nb):
            t = pipe.submit_host(h)
            if pending is not None:
                pipe.wait(pending)
            pending = t
        pipe.wait(pending)

    for pipe in arms.values():
        run(pipe)                                                        # warm-up: graph captures, first touch
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for name, pipe in arms.items():
            t0 = time.perf_counter()
            run(pipe)
            torch.cuda.synchronize()
            res[name].append(B * nb / (time.perf_counter() - t0))
    print(f"end to end: DewarpPipeline docs={B}, bf16x3, S=3, n_batch=2, {H}x{W} photos, submit_host/wait with two batches "
          f"outstanding, {nb} batches per run, {rounds} rounds alternating the arms")
    for name, pipe in arms.items():
        v = res[name]
        print(f"{name:28s} out {tuple(pipe.out_u8.shape)}  d2h {pipe.d2h_bytes / 1e6:6.1f} MB/batch  docs/s " +
              " ".join(f"{x:6.1f}" for x in v) + f"   mean {sum(v) / len(v):6.1f}")


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
