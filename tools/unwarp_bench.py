"""Standalone timing of the fused upsample+unwarp kernel.

CUDA events around N back-to-back launches that rotate over enough distinct (photo, output) buffer pairs to exceed the 126 MB
L2, so every launch reads its photo from HBM; the launches are replayed from one CUDA graph, so host launch latency is not in the number.
UW_AMP sets the synthetic map's amplitude (0.05 = the strongly warped default of the parity tests).

--mixed times the mixed-size uint8 launch (dvd_unwarp_u8_mixed) the same way: 16 documents cycling over eight photo sizes in ONE
launch vs 16 fixed-size launches with B = 1, and 16 x 1500x2000 in one mixed launch vs the batched fixed-size launch with B = 16."""
import os, subprocess, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import synth_workload as synth
from dvd_b200 import dewarp_fullres


MIXED_SIZES = [(1500, 2000), (2000, 1500), (4032, 3024), (3024, 4032), (1200, 1600), (1333, 999), (2448, 3264), (600, 450)]


def _timed_graph(launch, nbuf, n_launch):
    """us per launch of `launch(i)` (buffer set i % nbuf), n_launch launches replayed from one CUDA graph"""
    for i in range(nbuf):
        launch(i)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(n_launch):
            launch(i % nbuf)
    graph.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); graph.replay(); e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n_launch


def main_mixed():
    from dvd_b200 import _lib
    from dvd_b200.unwarp import AFFINE, plan_mixed, table_bytes
    dev = torch.device("cuda:0")
    l = _lib.lib()
    amp = float(os.environ.get("UW_AMP", "0.05"))
    n_launch = int(os.environ.get("UW_LAUNCHES", "60"))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"GPU: {q}", flush=True)
    for label, sizes in (("16 mixed sizes", [MIXED_SIZES[i % 8] for i in range(16)]), ("16 x 1500x2000", [(1500, 2000)] * 16)):
        maps = torch.cat([synth.make_map64(5 + i, "smooth", amp=amp) for i in range(16)]).to(dev)
        px = sum(H * W for H, W in sizes)
        nbuf = max(2, (400 << 20) // (6 * px) + 1)                 # >= 400 MB of distinct traffic before a buffer set repeats
        base = [synth.make_photo(H, W, 21 + k, "page")[0].permute(1, 2, 0).to(torch.uint8).contiguous() for k, (H, W) in enumerate(sizes)]
        photos = [[p.to(dev) for p in base] for _ in range(nbuf)]
        outs = [[torch.empty_like(p) for p in ph] for ph in photos]
        tables = []
        for b in range(nbuf):
            th = torch.empty(table_bytes(16), dtype=torch.uint8).pin_memory()
            plan_mixed(th, photos[b], outs[b], 64, 64)
            tables.append(th.to(dev))
        st = lambda: _lib.stream_ptr()
        t_mixed = _timed_graph(lambda b: _lib.check(l.dvd_unwarp_u8_mixed(_lib.ptr(tables[b]), 3, _lib.ptr(maps), st()), "mixed"), nbuf, n_launch)
        if label.startswith("16 x"):
            H, W = sizes[0]
            bat_in = [torch.stack(ph) for ph in photos]
            bat_out = [torch.empty_like(x) for x in bat_in]
            t_ref = _timed_graph(lambda b: _lib.check(l.dvd_unwarp_u8(_lib.ptr(bat_in[b]), _lib.ptr(maps), _lib.ptr(bat_out[b]), 16, 3, H, W,
                                                                      64, 64, AFFINE, st()), "u8"), nbuf, n_launch)
            ref_name = "one batched dvd_unwarp_u8 launch (B=16)"
        else:
            def per_doc(b):
                for k, ((H, W), p, o) in enumerate(zip(sizes, photos[b], outs[b])):
                    _lib.check(l.dvd_unwarp_u8(_lib.ptr(p), _lib.ptr(maps[k:k + 1]), _lib.ptr(o), 1, 3, H, W, 64, 64, AFFINE, st()), "u8")
            t_ref = _timed_graph(per_doc, nbuf, max(1, n_launch // 4))
            ref_name = "16 fixed-size launches (B=1)"
        for name, t in (("mixed launch", t_mixed), (ref_name, t_ref)):
            print(f"unwarp u8 {label} amp={amp}: {name:40s} {t:8.1f} us  {6 * px / t / 1e3:7.1f} GB/s (6 B/px, {px / 1e6:.1f} Mpx, "
                  f"{nbuf} buffer sets)", flush=True)
        print(f"  mixed / reference = {t_mixed / t_ref:.3f}", flush=True)
        del photos, outs, tables


def main():
    if "--mixed" in sys.argv:
        return main_mixed()
    dev = torch.device("cuda:0")
    amp = float(os.environ.get("UW_AMP", "0.05"))
    m = synth.make_map64(5, "smooth", amp=amp).to(dev)
    n_launch = int(os.environ.get("UW_LAUNCHES", "60"))
    for (H, W) in [(1500, 2000), (4032, 3024)]:
        photo = synth.make_photo(H, W, 21, "page").to(dev)
        pu8 = photo[0].permute(1, 2, 0).to(torch.uint8).unsqueeze(0).contiguous()
        for name, src, bpp in (("f32->f32", photo, 24), ("u8->u8", pu8, 6)):
            per = src.numel() * src.element_size() * 2
            nbuf = max(2, (400 << 20) // per + 1)                       # >= 400 MB of distinct traffic before a buffer repeats
            ins = [src.clone() for _ in range(nbuf)]
            outs = [torch.empty_like(src) for _ in range(nbuf)]
            for i in range(nbuf):
                dewarp_fullres(m, ins[i], out=outs[i])
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()                              # one graph of n_launch kernels: no host time between launches
            with torch.cuda.graph(graph):
                for i in range(n_launch):
                    dewarp_fullres(m, ins[i % nbuf], out=outs[i % nbuf])
            graph.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); graph.replay(); e1.record(); e1.synchronize()
            t = e0.elapsed_time(e1) * 1e3 / n_launch
            print(f"unwarp {name:9s} {W}x{H} amp={amp}: {t:7.1f} us  {bpp * H * W / t / 1e3:7.1f} GB/s ({bpp} B/px, {nbuf} buffer pairs)", flush=True)
            del ins, outs


if __name__ == "__main__":
    main()
