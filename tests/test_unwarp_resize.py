"""Dewarping to a requested output size: the sized uint8 HWC launch (dvd_unwarp_u8_sized_plan / dvd_unwarp_u8_sized), the size= form
of dewarp_fullres and DewarpPipeline(out_size=...).  The planner and the C layout are checked without a GPU; on the GPU the output
is compared with the fixed-size kernel (same size, s = 1) and with the float64 oracle
    trunc(avg_pool2d(grid_sample_ref(photo, fullres_grid(map64, s*Ho, s*Wo)), s))."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import synth

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
cdiv = lambda a, b: -(-a // b)


def _auto(H, W, Ho, Wo):
    return min(8, max(1, cdiv(H, Ho), cdiv(W, Wo)))


def _plan(docs, C_=3, table_bytes=None, ptrs=(0x1000, 0x2000), mh=64, mw=64):
    """docs: (H, W, Ho, Wo, supersample) tuples -> (rc, tiles, chosen factors, error message)"""
    from dvd_b200 import _lib
    l = _lib.lib()
    n = len(docs)
    arr = (_lib.SizedUnwarpDoc * max(n, 1))(*[_lib.SizedUnwarpDoc(ptrs[0], ptrs[1], H, W, Ho, Wo, s, 0) for H, W, Ho, Wo, s in docs])
    nb = l.dvd_unwarp_sized_table_bytes(n) if table_bytes is None else table_bytes
    table = C.create_string_buffer(max(nb, 1))
    tiles = C.c_longlong(-1)
    chosen = (C.c_int32 * max(n, 1))()
    rc = l.dvd_unwarp_u8_sized_plan(arr, n, C_, mh, mw, 0.987, table, nb, C.byref(tiles), chosen)
    return rc, tiles.value, list(chosen)[:n], l.dvd_last_error().decode()


AUTO_CASES = [  # H, W, Ho, Wo -> s
    (1500, 2000, 1500, 2000, 1), (1500, 2000, 3000, 4000, 1), (100, 100, 400, 50, 2),      # same size, upscaling, mixed
    (4032, 3024, 2016, 1512, 2), (4032, 3024, 1008, 756, 4), (4032, 3024, 504, 378, 8),    # exact ratios
    (4032, 3024, 2048, 1536, 2), (4032, 3024, 1024, 768, 4), (4032, 3024, 512, 384, 8),    # non-integer ratios
    (1000, 1000, 333, 1000, 4), (1000, 1000, 1000, 334, 3), (9, 7, 1, 1, 8),
    (4032, 3024, 100, 75, 8), (5000, 5000, 1, 1, 8), (3000, 100, 20, 100, 8),               # ratios above 8
]


def test_auto_supersample_factor_without_a_gpu():
    docs = [(H, W, Ho, Wo, 0) for H, W, Ho, Wo, _ in AUTO_CASES]
    rc, _, chosen, msg = _plan(docs)
    assert rc == 0, msg
    assert chosen == [s for *_, s in AUTO_CASES] == [_auto(*c[:4]) for c in AUTO_CASES]
    # explicit factors are kept as given
    rc, _, chosen, _ = _plan([(H, W, Ho, Wo, k % 8 + 1) for k, (H, W, Ho, Wo, _) in enumerate(AUTO_CASES)])
    assert rc == 0 and chosen == [k % 8 + 1 for k in range(len(AUTO_CASES))]


def test_plan_counts_tiles_and_empty_documents_without_a_gpu():
    docs = [(1500, 2000, 1500, 2000, 1), (1500, 2000, 750, 1000, 0), (4032, 3024, 1024, 768, 0), (7, 5, 33, 17, 1),
            (600, 450, 1, 1, 0), (10, 10, 0, 10, 0), (0, 10, 10, 10, 3), (10, 0, 10, 10, 0), (10, 10, 10, 0, 0), (600, 450, 257, 129, 3)]
    rc, tiles, chosen, msg = _plan(docs)
    assert rc == 0, msg
    want = 0
    for (H, W, Ho, Wo, _), s in zip(docs, chosen):
        if 0 in (H, W, Ho, Wo):
            continue
        want += cdiv(Wo, 128) * cdiv(Ho, 8) if s == 1 else cdiv(Wo, 32) * cdiv(Ho, 8)
    assert tiles == want
    assert chosen[5:9] == [1, 3, 1, 1]                           # empty documents: auto -> 1, explicit kept
    assert _plan([])[:2] == (0, 0)
    # empty documents may have null pointers
    assert _plan([(0, 10, 5, 5, 0), (10, 10, 0, 5, 0)], ptrs=(0, 0))[0] == 0


ERRORS = {  # case -> (_plan kwargs, message fragment)
    "C0": (dict(C_=0), "C=0 outside 1..4"), "C5": (dict(C_=5), "C=5 outside 1..4"),
    "negative_photo": (dict(docs=[(10, 10, 5, 5, 0), (-1, 10, 5, 5, 0)]), "document 1 has a negative size"),
    "negative_output": (dict(docs=[(10, 10, 5, -5, 0)]), "document 0 has a negative size"),
    "supersample_neg": (dict(docs=[(10, 10, 5, 5, -1)]), "supersample=-1 outside 0..8"),
    "supersample_9": (dict(docs=[(10, 10, 5, 5, 9)]), "supersample=9 outside 0..8"),
    "photo_too_large": (dict(docs=[(32768, 21846, 10, 10, 0)]), "photo (32768x21846x3) is too large"),
    "output_too_large": (dict(docs=[(10, 10, 32768, 21846, 0)]), "output (32768x21846x3) is too large"),
    "null_photo": (dict(ptrs=(0, 0x2000)), "null photo or output pointer"),
    "null_out": (dict(ptrs=(0x1000, 0)), "null photo or output pointer"),
    "table_too_small": (dict(table_bytes=-1), "is too small for 2 documents"),
    "map_size": (dict(mh=0), "bad map size 0x64"),
    "map_size_large": (dict(mw=65536), "bad map size 64x65536"),
    "too_many_tiles": (dict(docs=[(8, 8, 46340, 46340, 2)] * 130, C_=1), "more than 1073741824 tiles"),
}


@pytest.mark.parametrize("case", sorted(ERRORS))
def test_plan_rejects_bad_input(case):
    from dvd_b200 import _lib
    kw, frag = dict(ERRORS[case][0]), ERRORS[case][1]
    docs = kw.pop("docs", [(10, 10, 5, 5, 0), (20, 30, 40, 60, 1)])
    if kw.get("table_bytes") == -1:
        kw["table_bytes"] = _lib.lib().dvd_unwarp_sized_table_bytes(len(docs)) - 1
    rc, _, _, msg = _plan(docs, **kw)
    assert rc == -1 and msg.startswith("unwarp_u8_sized_plan") and frag in msg, (rc, msg)


def test_sized_doc_layout_matches_c(tmp_path):
    from dvd_b200 import _lib
    fields = ["photo", "out", "H", "W", "Ho", "Wo", "supersample", "pad"]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvd_b200.h"\nint main(){printf("%zu' + " %zu" * len(fields) +
                   '\\n",sizeof(dvd_unwarp_sized_doc_t)' + "".join(f",offsetof(dvd_unwarp_sized_doc_t,{f})" for f in fields) +
                   ');return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = _lib.SizedUnwarpDoc
    assert got == [C.sizeof(D)] + [getattr(D, f).offset for f in fields]


def test_dewarp_fullres_rejects_bad_size_arguments_without_a_gpu():
    """argument checks that run before any CUDA call"""
    from dvd_b200.unwarp import size_arg, supersample_arg
    assert supersample_arg("auto") == 0 and [supersample_arg(k) for k in range(1, 9)] == list(range(1, 9))
    for bad in (0, 9, -1, "2", 2.0, True, None):
        with pytest.raises(ValueError):
            supersample_arg(bad)
    assert size_arg((3, 4)) == (3, 4)
    for bad in ((0, 4), (4, -1), (4,), (1, 2, 3), "4x4", (2.0, 3), None, (True, 2)):
        with pytest.raises(ValueError):
            size_arg(bad)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dvd_b200 import _lib
    _lib.check(_lib.lib().dvd_check_device(), "dvd_check_device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def model(dev, state_dict_live):
    from dvd_b200.model import DiT
    m = DiT(precision="fp32")
    m.load_state_dict(state_dict_live, strict=False)
    return m.to(dev).eval()


def _rotation_map(deg, zoom=1.0):
    t = np.deg2rad(deg)
    ys, xs = torch.meshgrid(torch.linspace(0, 1, 64), torch.linspace(0, 1, 64), indexing="ij")
    cx, cy = xs - 0.5, ys - 0.5
    rx = zoom * (np.cos(t) * cx - np.sin(t) * cy) + 0.5
    ry = zoom * (np.sin(t) * cx + np.cos(t) * cy) + 0.5
    return torch.stack([rx - xs, ry - ys])[None].float().contiguous()


def _maps(kind, n):
    if kind == "smooth":
        return torch.cat([synth.make_map64(40 + i, "smooth") for i in range(n)])
    if kind == "rotation":
        return torch.cat([_rotation_map(-20.0 + 7.0 * i, 1.0 + 0.05 * (i % 3)) for i in range(n)])
    return torch.cat([synth.make_map64(60 + i, "adversarial") for i in range(n)])         # white noise


def _photo(H, W, seed, kind="noise", C_=3):
    """uint8 HWC photo with C_ channels (page or noise content)"""
    p = synth.make_photo(H, W, seed, kind)[0].permute(1, 2, 0).to(torch.uint8)
    if C_ <= 3:
        return p[..., :C_].contiguous()
    return torch.cat([p, p[..., :1].flip(0)], dim=2).contiguous()


def _sized(maps, photos, outs, supersample=0):
    """one sized launch through the C ABI (photos [H,W,C] / outs [Ho,Wo,C] device tensors); returns the chosen factors"""
    from dvd_b200 import _lib
    from dvd_b200.unwarp import plan_sized, sized_table_bytes
    th = torch.empty(sized_table_bytes(len(photos)), dtype=torch.uint8).pin_memory()
    _, chosen = plan_sized(th, photos, outs, 64, 64, supersample, C=photos[0].shape[2])
    table = th.to(maps.device)
    _lib.check(_lib.lib().dvd_unwarp_u8_sized(_lib.ptr(table), photos[0].shape[2], _lib.ptr(maps), _lib.stream_ptr()), "sized")
    torch.cuda.synchronize()
    return chosen


def _oracle(map1, photo_hwc, Ho, Wo, s):
    """float64 reference: trunc(avg_pool2d(grid_sample_ref(photo, fullres_grid(map, s*Ho, s*Wo)), s)) as uint8 HWC (CPU)"""
    from oracle import dvd_oracle as O
    ph = photo_hwc.cpu().permute(2, 0, 1)[None].double()
    ref = O.grid_sample_ref(ph, O.fullres_grid(map1.cpu().double(), s * Ho, s * Wo))
    if s > 1:
        ref = torch.nn.functional.avg_pool2d(ref, s)
    return ref[0].permute(1, 2, 0).clamp(0, 255)


def _check_oracle(got, ref):
    diff = (got.cpu().double() - torch.floor(ref)).abs()
    assert float(diff.max()) <= 1, float(diff.max())
    mse = float(((got.cpu().double() - ref) ** 2).mean())
    psnr = 10 * np.log10(255.0 ** 2 / max(mse, 1e-12))
    assert psnr >= 45.0, psnr


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["smooth", "rotation", "noise"])
@pytest.mark.parametrize("C_", [1, 3, 4])
def test_same_size_s1_is_byte_equal_to_fixed_launch(dev, kind, C_):
    """size == photo size with s = 1: byte-equal to dvd_unwarp_u8, for the fast and general bodies, W not a multiple of 4 or 128"""
    from dvd_b200 import dewarp_fullres
    sizes = [(1500, 2000), (1333, 999), (600, 450), (9, 130), (7, 5), (1, 640), (250, 131)]
    maps = _maps(kind, len(sizes)).to(dev)
    photos = [_photo(H, W, 500 + i, "page" if i % 2 else "noise", C_).to(dev) for i, (H, W) in enumerate(sizes)]
    outs = [torch.full_like(p, 7) for p in photos]
    assert _sized(maps, photos, outs, 1) == [1] * len(sizes)
    for i, (p, o) in enumerate(zip(photos, outs)):
        assert torch.equal(o, dewarp_fullres(maps[i:i + 1], p.unsqueeze(0))[0]), sizes[i]
    # auto picks s = 1 at the photo's size
    outs2 = [torch.empty_like(p) for p in photos]
    assert _sized(maps, photos, outs2, 0) == [1] * len(sizes)
    assert all(torch.equal(a, b) for a, b in zip(outs, outs2))


S1_CASES = [(240, 320, 120, 160), (240, 320, 97, 211), (120, 90, 300, 260), (200, 150, 150, 200), (64, 80, 1, 57),
            (64, 80, 45, 1), (64, 80, 1, 1), (150, 200, 37, 700)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["smooth", "rotation", "noise"])
def test_s1_other_sizes_match_oracle(dev, kind):
    maps = _maps(kind, len(S1_CASES)).to(dev)
    photos = [_photo(H, W, 600 + i, "page" if i % 2 else "noise").to(dev) for i, (H, W, _, _) in enumerate(S1_CASES)]
    outs = [torch.empty((Ho, Wo, 3), dtype=torch.uint8, device=dev) for _, _, Ho, Wo in S1_CASES]
    _sized(maps, photos, outs, 1)
    for i, ((H, W, Ho, Wo), p, o) in enumerate(zip(S1_CASES, photos, outs)):
        _check_oracle(o, _oracle(maps[i:i + 1], p, Ho, Wo, 1))


SS_CASES = [  # H, W, Ho, Wo, s (0 = auto)
    (240, 320, 120, 160, 2), (240, 320, 80, 107, 3), (240, 320, 60, 80, 4), (240, 320, 48, 64, 5), (240, 320, 30, 40, 8),
    (240, 320, 61, 77, 0), (300, 200, 37, 29, 0), (100, 140, 1, 9, 0), (100, 140, 13, 1, 5), (90, 130, 45, 65, 0),
    (200, 300, 200, 300, 2), (50, 60, 80, 40, 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["smooth", "rotation", "noise"])
def test_supersampled_sizes_match_oracle(dev, kind):
    from dvd_b200.unwarp import plan_sized, sized_table_bytes
    maps = _maps(kind, len(SS_CASES)).to(dev)
    photos = [_photo(H, W, 700 + i, "page" if i % 2 else "noise").to(dev) for i, (H, W, *_) in enumerate(SS_CASES)]
    outs = [torch.empty((Ho, Wo, 3), dtype=torch.uint8, device=dev) for _, _, Ho, Wo, _ in SS_CASES]
    chosen = _sized(maps, photos, outs, [c[4] for c in SS_CASES])
    assert chosen == [c[4] or _auto(*c[:4]) for c in SS_CASES]
    for i, ((H, W, Ho, Wo, _), p, o) in enumerate(zip(SS_CASES, photos, outs)):
        _check_oracle(o, _oracle(maps[i:i + 1], p, Ho, Wo, chosen[i]))
    # the planner reports the factor it used
    th = torch.empty(sized_table_bytes(len(photos)), dtype=torch.uint8)
    assert plan_sized(th, photos, outs, 64, 64, 0)[1] == [_auto(*c[:4]) for c in SS_CASES]


@pytest.mark.gpu
def test_mixed_batch_equals_single_document_launches(dev):
    """different photo sizes, output sizes and factors in one launch: each document equals its own one-document launch, and canary
    bytes around and between the outputs in one arena stay untouched"""
    from dvd_b200.pipeline import DewarpPipeline
    docs = [(1500, 2000, 750, 1000, 0), (1333, 999, 1333, 999, 1), (600, 450, 100, 75, 0), (7, 5, 30, 20, 1), (4032, 3024, 504, 378, 0),
            (250, 131, 97, 61, 3), (9, 130, 3, 40, 0), (640, 480, 2048, 1536, 0)]
    maps = _maps("rotation", len(docs)).to(dev)
    photos = [_photo(H, W, 800 + i, "page").to(dev) for i, (H, W, *_) in enumerate(docs)]
    shapes = [(Ho, Wo, 3) for _, _, Ho, Wo, _ in docs]
    total = sum(Ho * Wo * 3 + 16 for Ho, Wo, _ in shapes) + 64
    arena = torch.full((total,), 0x5A, dtype=torch.uint8, device=dev)
    outs = DewarpPipeline._arena_views(arena[32:], shapes)
    chosen = _sized(maps, photos, outs, [d[4] for d in docs])
    written = torch.zeros(total, dtype=torch.bool, device=dev)
    for o in outs:
        off = o.data_ptr() - arena.data_ptr()
        written[off:off + o.numel()] = True
    assert bool((arena[~written] == 0x5A).all())
    for i, (p, o) in enumerate(zip(photos, outs)):
        one = torch.empty_like(o)
        assert _sized(maps[i:i + 1], [p], [one], chosen[i]) == [chosen[i]]
        assert torch.equal(o, one), docs[i]


@pytest.mark.gpu
def test_sized_graph_serves_a_new_composition(dev):
    from dvd_b200 import _lib
    from dvd_b200.unwarp import plan_sized, sized_table_bytes
    maps = _maps("smooth", 3).to(dev)
    pa = [_photo(H, W, 900 + i).to(dev) for i, (H, W) in enumerate([(1500, 2000), (600, 450), (9, 130)])]
    oa = [torch.empty((Ho, Wo, 3), dtype=torch.uint8, device=dev) for Ho, Wo in [(500, 666), (600, 450), (2, 65)]]
    pb = [_photo(H, W, 950 + i).to(dev) for i, (H, W) in enumerate([(1333, 999), (7, 5)])]
    ob = [torch.empty((Ho, Wo, 3), dtype=torch.uint8, device=dev) for Ho, Wo in [(333, 250), (70, 50)]]
    want_a = [torch.empty_like(o) for o in oa]
    want_b = [torch.empty_like(o) for o in ob]
    _sized(maps, pa, want_a)
    _sized(maps[:2], pb, want_b)
    th = torch.empty(sized_table_bytes(3), dtype=torch.uint8).pin_memory()
    table = torch.empty(sized_table_bytes(3), dtype=torch.uint8, device=dev)
    plan_sized(th, pa, oa, 64, 64, 0)
    table.copy_(th)
    launch = lambda: _lib.check(_lib.lib().dvd_unwarp_u8_sized(_lib.ptr(table), 3, _lib.ptr(maps), _lib.stream_ptr()), "sized")
    launch(); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for o in oa:
        o.fill_(0xAB)
    g.replay(); torch.cuda.synchronize()
    assert all(torch.equal(o, w) for o, w in zip(oa, want_a))
    for o in oa:
        o.fill_(0xAB)
    plan_sized(th, pb, ob, 64, 64, 0)
    table.copy_(th)
    g.replay(); torch.cuda.synchronize()
    assert all(torch.equal(o, w) for o, w in zip(ob, want_b))
    assert all(bool((o == 0xAB).all()) for o in oa)
    # a table planned for another C writes nothing
    for o in ob:
        o.fill_(0xCD)
    _lib.check(_lib.lib().dvd_unwarp_u8_sized(_lib.ptr(table), 4, _lib.ptr(maps), _lib.stream_ptr()), "sized")
    torch.cuda.synchronize()
    assert all(bool((o == 0xCD).all()) for o in ob)


@pytest.mark.gpu
def test_dewarp_fullres_size(dev):
    from dvd_b200 import dewarp_fullres
    maps = _maps("rotation", 3).to(dev)
    batch = torch.stack([_photo(300, 400, 1000 + i) for i in range(3)]).to(dev)
    for size, ss in (((150, 200), "auto"), ((75, 100), 4), ((300, 400), 1), ((500, 90), "auto")):
        got = dewarp_fullres(maps, batch, size=size, supersample=ss)
        assert got.shape == (3,) + size + (3,) and got.dtype == torch.uint8
        for i in range(3):
            one = torch.empty(size + (3,), dtype=torch.uint8, device=dev)
            _sized(maps[i:i + 1], [batch[i]], [one], 0 if ss == "auto" else ss)
            assert torch.equal(got[i], one)
        out = torch.empty_like(got)
        assert dewarp_fullres(maps, batch, out=out, size=size, supersample=ss) is out and torch.equal(out, got)
    assert torch.equal(dewarp_fullres(maps, batch, size=(300, 400), supersample=1), dewarp_fullres(maps, batch))
    # list form: one size for all, or one per photo
    photos = [_photo(H, W, 1100 + i).to(dev) for i, (H, W) in enumerate([(300, 400), (123, 77), (640, 480)])]
    outs = dewarp_fullres(maps, photos, size=(60, 80))
    assert [tuple(o.shape) for o in outs] == [(60, 80, 3)] * 3
    sizes = [(150, 200), (123, 77), (80, 60)]
    outs = dewarp_fullres(maps, photos, size=sizes, supersample=2)
    for i, (p, o) in enumerate(zip(photos, outs)):
        one = torch.empty(sizes[i] + (3,), dtype=torch.uint8, device=dev)
        _sized(maps[i:i + 1], [p], [one], 2)
        assert torch.equal(o, one)
    assert dewarp_fullres(maps[:0], [], size=(4, 4)) == []
    for kw in (dict(photo=batch.permute(0, 3, 1, 2).float(), size=(10, 10)), dict(size=(0, 10)), dict(size=(10,)),
               dict(size=(10, 10), supersample=0), dict(size=(10, 10), supersample=9), dict(size=(10, 10), supersample="x"),
               dict(photo=photos, size=[(10, 10)] * 2), dict(photo=photos, size=[(10, 10), (10, 10), (0, 1)])):
        kw.setdefault("photo", batch)
        with pytest.raises(ValueError):
            dewarp_fullres(maps, **kw)


KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")


def _docs(sizes):
    docs = []
    for i, (H, W) in enumerate(sizes):
        d = synth.make_doc_inputs(i, H=H, W=W)
        d["photo_u8"] = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous()
        docs.append(d)
    return docs


@pytest.mark.gpu
def test_pipeline_fixed_out_size(dev, model, monkeypatch):
    from dvd_b200 import dewarp_fullres
    from dvd_b200.pipeline import DewarpPipeline
    captures = []
    real_graph = torch.cuda.graph
    monkeypatch.setattr(torch.cuda, "graph", lambda *a, **k: (captures.append(1), real_graph(*a, **k))[1])
    H, W, out = 120, 160, (50, 70)
    pipe = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=2, height=H, width=W, out_size=out)
    assert pipe.out_u8.shape == (2,) + out + (3,) and pipe.d2h_bytes == 2 * 50 * 70 * 3
    batches = [_docs([(H, W)] * 2), [synth.make_doc_inputs(7 + i, H=H, W=W) for i in range(2)]]
    for d in batches[1]:
        d["photo_u8"] = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous()
    hs = []
    for docs in batches:
        h = {k: torch.cat([d[k] for d in docs]).contiguous().pin_memory() for k in KEYS}
        h["photo_u8"] = torch.stack([d["photo_u8"] for d in docs]).pin_memory()
        hs.append(h)

    def want(h):
        return dewarp_fullres(pipe.map64, h["photo_u8"].to(dev), size=out).cpu()
    for h in hs:
        got = pipe.run_host(h).clone()
        assert got.shape == (2,) + out + (3,) and torch.equal(got, want(h))
    n_caps = len(captures)
    tickets, got = [], []
    for i, h in enumerate(hs + hs):
        tickets.append(pipe.submit_host(h))
        if i >= 1:
            got.append(pipe.wait(tickets[i - 1]).clone())
    got.append(pipe.wait(tickets[-1]).clone())
    assert len(captures) == n_caps
    for g, h in zip(got, hs + hs):
        assert torch.equal(g, pipe.run_host(h))
    dset = {k: v.to(dev) for k, v in hs[0].items()}
    for _ in range(2):
        assert torch.equal(pipe.run_device(dset), dewarp_fullres(pipe.map64, dset["photo_u8"], size=out))
    # callable out_size, explicit factor
    pipe2 = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=2, height=H, width=W, out_size=lambda h, w: (h // 3, w // 3),
                           supersample=2)
    got = pipe2.run_host(hs[1])
    assert torch.equal(got, dewarp_fullres(pipe2.map64, hs[1]["photo_u8"].to(dev), size=(40, 53), supersample=2).cpu())


@pytest.mark.gpu
def test_pipeline_mixed_out_size(dev, model, monkeypatch):
    from dvd_b200 import dewarp_fullres
    from dvd_b200.pipeline import DewarpPipeline
    sizes = [(96, 128), (64, 200), (120, 90), (72, 72)]
    docs = _docs(sizes)
    long_side = lambda H, W: (max(1, round(H * 48 / max(H, W))), max(1, round(W * 48 / max(H, W))))
    captures = []
    real_graph = torch.cuda.graph
    monkeypatch.setattr(torch.cuda, "graph", lambda *a, **k: (captures.append(1), real_graph(*a, **k))[1])
    P = sum(H * W for H, W in sizes[:3])
    pipe = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=3, max_pixels=P, out_size=long_side)
    assert pipe.d2h_bytes == 3 * P + 16 * 3

    def batch(ds):
        h = {k: torch.cat([d[k] for d in ds]).contiguous().pin_memory() for k in KEYS}
        h["photo_u8"] = [d["photo_u8"].pin_memory() for d in ds]
        return h

    def check(got, ds):
        assert len(got) == len(ds)
        for i, (g, d) in enumerate(zip(got, ds)):
            H, W = d["photo_u8"].shape[:2]
            assert tuple(g.shape) == long_side(H, W) + (3,)
            want = dewarp_fullres(pipe.map64[i:i + 1], [d["photo_u8"].to(dev)], size=long_side(H, W))[0]
            assert torch.equal(g.to(dev), want)
    for sel in ([0, 1, 2], [3], [2, 0], [1, 3, 0]):
        ds = [docs[i] for i in sel]
        check([g.clone() for g in pipe.run_host(batch(ds))], ds)
    n_caps = len(captures)
    assert n_caps == 4
    seq = [[0, 1, 2], [3], [2, 0], [1, 3, 0]]
    tickets, outs = [], []
    for i, sel in enumerate(seq):
        tickets.append(pipe.submit_host(batch([docs[j] for j in sel])))
        if i >= 1:
            outs.append([g.clone() for g in pipe.wait(tickets[i - 1])])
    outs.append([g.clone() for g in pipe.wait(tickets[-1])])
    assert len(captures) == n_caps
    for got, sel in zip(outs, seq):
        assert all(torch.equal(x, y) for x, y in zip(got, pipe.run_host(batch([docs[j] for j in sel]))))
    full = docs[:3]
    dset = {k: v.to(dev) for k, v in batch(full).items() if k != "photo_u8"}
    dset["photo_u8"] = [d["photo_u8"].to(dev) for d in full]
    for _ in range(2):
        check([g.clone() for g in pipe.run_device(dset)], full)
    dset["photo_u8"] = [docs[3]["photo_u8"].to(dev), docs[0]["photo_u8"].to(dev), docs[1]["photo_u8"].to(dev)]
    n_caps = len(captures)
    got = pipe.run_device(dset)
    assert len(captures) == n_caps
    for i, g in enumerate(got):
        H, W = dset["photo_u8"][i].shape[:2]
        assert torch.equal(g, dewarp_fullres(pipe.map64[i:i + 1], [dset["photo_u8"][i]], size=long_side(H, W))[0])
    # outputs past max_out_pixels
    small = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=3, max_pixels=P, out_size=(60, 60), max_out_pixels=3 * 3600 - 1)
    with pytest.raises(ValueError):
        small.run_host(batch(docs[:3]))
    with pytest.raises(ValueError):
        small.run_device(dict(dset))
    assert len(small.run_host(batch(docs[:2]))) == 2
    with pytest.raises(ValueError):
        DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=1, out_size=(0, 5))
    with pytest.raises(ValueError):
        DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=1, out_size=(5, 5), supersample=9)
