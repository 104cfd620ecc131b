"""Standalone timing of the decoder's depthwise 3x3 convolution of the tensor modes (dvd_test_dwconv: bf16 pair in, bf16 pair out, C = 2048).

CUDA events around one CUDA graph of back-to-back launches, so host launch latency is not in the number.  Two cases:
  N = 2  (one document, two hypotheses): the same 16.8 MB input every launch, so it is read from L2 as inside a denoiser step, where
         conv1 has just written it;
  N = 32 (16 documents in flight): 268 MB in and 268 MB out, more than the 126 MB L2, so the launch streams from HBM.
GB/s counts the compulsory traffic: the input pair read once and the output pair written once, N/2 x 33.6 MB.
Usage: python tools/dwconv_bench.py [--launches 40] [--n 2 32]"""
import argparse, os, subprocess, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dvd_b200 import _lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=40)
    ap.add_argument("--n", type=int, nargs="+", default=[2, 32])
    a = ap.parse_args()
    if a.launches < 20:
        ap.error("--launches must be at least 20")
    dev = torch.device("cuda:0")
    l = _lib.lib()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    print(f"GPU: {q.strip()}", flush=True)
    C = 2048
    g = torch.Generator(device=dev).manual_seed(0)
    w9 = torch.randn(9, C, device=dev, generator=g) * 0.3
    scale = torch.rand(C, device=dev, generator=g) + 0.5
    shift = torch.randn(C, device=dev, generator=g) * 0.1
    for N in a.n:
        x = torch.randn(N, 1024, C, device=dev, generator=g)
        hi = x.to(torch.bfloat16)
        lo = (x - hi.float()).to(torch.bfloat16)
        del x
        out_hi, out_lo = torch.empty_like(hi), torch.empty_like(hi)

        def launch():
            _lib.check(l.dvd_test_dwconv(_lib.ptr(hi), _lib.ptr(lo), _lib.ptr(w9), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(out_hi),
                                         _lib.ptr(out_lo), N, C, _lib.stream_ptr()), "dvd_test_dwconv")

        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            launch()                                    # module load, shared-memory opt-in
            s.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=s):
                for _ in range(a.launches):
                    launch()
            graph.replay()
            s.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            times = []
            for _ in range(5):
                e0.record(s); graph.replay(); e1.record(s); e1.synchronize()
                times.append(e0.elapsed_time(e1) * 1e3 / a.launches)
        times.sort()
        us = times[len(times) // 2]
        nbytes = N * 1024 * C * 2 * 4                   # hi + lo in, hi + lo out
        print(f"dwconv N={N:3d} C={C}: {us:8.2f} us per launch (median of 5 replays of {a.launches}; min {times[0]:.2f} max {times[-1]:.2f})  "
              f"{nbytes / us / 1e3:8.1f} GB/s ({nbytes / 1e6:.1f} MB compulsory)", flush=True)
        del hi, lo, out_hi, out_lo, graph


if __name__ == "__main__":
    main()
