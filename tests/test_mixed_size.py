"""Mixed-size batches: the one-launch uint8 HWC unwarp of documents of different sizes (dvd_unwarp_u8_plan / dvd_unwarp_u8_mixed),
the list form of dewarp_fullres and DewarpPipeline(max_pixels=...).  The planner and the C layout are checked without a GPU;
everything else compares against the fixed-size kernel on each document alone."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
cdiv = lambda a, b: -(-a // b)


def _plan(shapes, C_=3, table_bytes=None, ptrs=(0x1000, 0x2000), mh=64, mw=64):
    from dvd_b200 import _lib
    l = _lib.lib()
    n = len(shapes)
    docs = (_lib.UnwarpDoc * max(n, 1))(*[_lib.UnwarpDoc(ptrs[0], ptrs[1], H, W) for H, W in shapes])
    nb = l.dvd_unwarp_table_bytes(n) if table_bytes is None else table_bytes
    table = C.create_string_buffer(max(nb, 1))
    tiles = C.c_longlong(-1)
    rc = l.dvd_unwarp_u8_plan(docs, n, C_, mh, mw, 0.987, table, nb, C.byref(tiles))
    return rc, tiles.value, l.dvd_last_error().decode()


def test_plan_counts_tiles_without_a_gpu():
    shapes = [(1500, 2000), (2000, 1500), (4032, 3024), (1333, 999), (600, 450), (1, 640), (7, 5), (9, 130), (0, 50), (50, 0)]
    rc, tiles, _ = _plan(shapes)
    assert rc == 0
    assert tiles == sum(cdiv(W, 128) * cdiv(H, 8) for H, W in shapes)
    assert _plan([])[:2] == (0, 0)


@pytest.mark.parametrize("case", ["table_too_small", "negative", "C0", "C5", "too_large", "null_photo", "null_out"])
def test_plan_rejects_bad_input(case):
    from dvd_b200 import _lib
    kw = {"table_too_small": dict(table_bytes=_lib.lib().dvd_unwarp_table_bytes(2) - 1),
          "negative": dict(shapes=[(10, 10), (-1, 10)]), "C0": dict(C_=0), "C5": dict(C_=5),
          "too_large": dict(shapes=[(10, 10), (32768, 21846)]), "null_photo": dict(ptrs=(0, 0x2000)),
          "null_out": dict(ptrs=(0x1000, 0))}[case]
    shapes = kw.pop("shapes", [(10, 10), (20, 30)])
    rc, _, msg = _plan(shapes, **kw)
    assert rc == -1 and msg.startswith("unwarp_u8_plan"), (rc, msg)
    # empty documents may have null pointers
    if case.startswith("null"):
        assert _plan([(0, 10), (10, 0)], **kw)[0] == 0


def test_unwarp_doc_layout_matches_c(tmp_path):
    from dvd_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvd_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                   'sizeof(dvd_unwarp_doc_t),offsetof(dvd_unwarp_doc_t,photo),offsetof(dvd_unwarp_doc_t,out),'
                   'offsetof(dvd_unwarp_doc_t,H),offsetof(dvd_unwarp_doc_t,W));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = _lib.UnwarpDoc
    assert got == [C.sizeof(D), D.photo.offset, D.out.offset, D.H.offset, D.W.offset]


# ---------------------------------------------------------------------------------------------------------------- GPU
SIZES = [(1500, 2000), (2000, 1500), (4032, 3024), (1333, 999), (600, 450), (1, 640), (7, 5), (9, 130)]


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


def _photo(H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randint(0, 256, (H, W, 3), generator=g, dtype=torch.uint8)


def _mixed(maps, photos, outs):
    """one mixed launch through the C ABI (photos / outs: device tensors [H,W,3])"""
    from dvd_b200 import _lib
    from dvd_b200.unwarp import plan_mixed, table_bytes
    th = torch.empty(table_bytes(len(photos)), dtype=torch.uint8).pin_memory()
    plan_mixed(th, photos, outs, 64, 64)
    table = th.to(maps.device)
    _lib.check(_lib.lib().dvd_unwarp_u8_mixed(_lib.ptr(table), 3, _lib.ptr(maps), _lib.stream_ptr()), "dvd_unwarp_u8_mixed")
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["smooth", "rotation", "noise"])
@pytest.mark.parametrize("layout", ["tensors", "arena"])
def test_mixed_kernel_is_byte_equal_to_fixed_launch(dev, kind, layout):
    """Every document of one mixed launch equals dvd_unwarp_u8 on that document alone, byte for byte, for fast-body shapes and the
    general body (narrower than 573 px or one row high), partial tiles on both axes and rows that are not a multiple of 16 bytes."""
    from dvd_b200 import dewarp_fullres
    maps = _maps(kind, len(SIZES)).to(dev)
    photos_h = [_photo(H, W, 100 + i) for i, (H, W) in enumerate(SIZES)]
    if layout == "tensors":
        photos = [p.to(dev) for p in photos_h]
        outs = [torch.full_like(p, 7) for p in photos]
    else:                                                        # views into one arena at 16-byte aligned offsets
        from dvd_b200.pipeline import DewarpPipeline
        total = sum(p.numel() + 16 for p in photos_h)
        parena = torch.zeros(total, dtype=torch.uint8, device=dev)
        oarena = torch.full((total,), 7, dtype=torch.uint8, device=dev)
        photos = DewarpPipeline._arena_views(parena, photos_h)
        outs = DewarpPipeline._arena_views(oarena, photos_h)
        for d, s in zip(photos, photos_h):
            d.copy_(s)
    _mixed(maps, photos, outs)
    for i, (p, o) in enumerate(zip(photos, outs)):
        want = dewarp_fullres(maps[i:i + 1], p.unsqueeze(0).contiguous())[0]
        assert torch.equal(o, want), (SIZES[i], int((o.int() - want.int()).abs().max()))


@pytest.mark.gpu
def test_mixed_kernel_matches_oracle(dev):
    from oracle import dvd_oracle as O
    m = _rotation_map(9.0, 1.1) + 0.3 * synth.make_map64(9, "smooth")
    photo = synth.make_photo(90, 130, 31, "noise")
    pu8 = photo[0].permute(1, 2, 0).to(torch.uint8).contiguous().to(dev)
    out = torch.empty_like(pu8)
    _mixed(m.to(dev), [pu8], [out])
    ref = O.unwarp(m, photo)[0].permute(1, 2, 0).clamp(0, 255)
    assert int((out.cpu().int() - ref.int()).abs().max()) <= 1


@pytest.mark.gpu
def test_mixed_graph_serves_a_new_composition(dev):
    """A launch captured once replays correctly after a different, smaller composition is planned into the same device table,
    and writes nothing into output buffers outside the batch."""
    from dvd_b200 import _lib, dewarp_fullres
    from dvd_b200.unwarp import plan_mixed, table_bytes
    sizes_a, sizes_b = [(1500, 2000), (600, 450), (9, 130)], [(1333, 999), (7, 5)]
    maps = _maps("smooth", 3).to(dev)
    pa = [_photo(H, W, 200 + i).to(dev) for i, (H, W) in enumerate(sizes_a)]
    pb = [_photo(H, W, 300 + i).to(dev) for i, (H, W) in enumerate(sizes_b)]
    oa, ob = [torch.empty_like(p) for p in pa], [torch.empty_like(p) for p in pb]
    th = torch.empty(table_bytes(3), dtype=torch.uint8).pin_memory()
    table = torch.empty(table_bytes(3), dtype=torch.uint8, device=dev)
    plan_mixed(th, pa, oa, 64, 64)
    table.copy_(th)
    launch = lambda: _lib.check(_lib.lib().dvd_unwarp_u8_mixed(_lib.ptr(table), 3, _lib.ptr(maps), _lib.stream_ptr()), "mixed")
    launch(); torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for o in oa:
        o.fill_(0xAB)
    g.replay(); torch.cuda.synchronize()
    for i, (p, o) in enumerate(zip(pa, oa)):
        assert torch.equal(o, dewarp_fullres(maps[i:i + 1], p.unsqueeze(0))[0])
    for o in oa:
        o.fill_(0xAB)
    plan_mixed(th, pb, ob, 64, 64)
    table.copy_(th)
    g.replay(); torch.cuda.synchronize()
    for i, (p, o) in enumerate(zip(pb, ob)):
        assert torch.equal(o, dewarp_fullres(maps[i:i + 1], p.unsqueeze(0))[0])
    for o in oa:                                                 # canaries: buffers of the earlier composition are untouched
        assert bool((o == 0xAB).all())


@pytest.mark.gpu
def test_dewarp_fullres_list_form(dev):
    from dvd_b200 import dewarp_fullres
    maps = _maps("rotation", 4).to(dev)
    photos = [_photo(H, W, 400 + i).to(dev) for i, (H, W) in enumerate([(600, 450), (1333, 999), (7, 5), (1500, 2000)])]
    outs = dewarp_fullres(maps, photos)
    assert isinstance(outs, list) and len(outs) == 4
    for i, (p, o) in enumerate(zip(photos, outs)):
        assert torch.equal(o, dewarp_fullres(maps[i:i + 1], p.unsqueeze(0))[0])
    assert dewarp_fullres(maps[:0], []) == []
    with pytest.raises(ValueError):
        dewarp_fullres(maps[:1], [photos[0].float()])


KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")
PIPE_SIZES = [(96, 128), (64, 200), (120, 90), (72, 72)]


def _host_docs():
    docs = []
    for i, (H, W) in enumerate(PIPE_SIZES):
        d = synth.make_doc_inputs(i, H=H, W=W)
        d["photo_u8"] = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous()
        docs.append(d)
    return docs


def _batch(docs):
    h = {k: torch.cat([d[k] for d in docs]).contiguous().pin_memory() for k in KEYS}
    h["photo_u8"] = [d["photo_u8"].pin_memory() for d in docs]
    return h


@pytest.mark.gpu
def test_pipeline_mixed_size(dev, model, monkeypatch):
    from dvd_b200 import dewarp_fullres
    from dvd_b200.pipeline import DewarpPipeline
    docs = _host_docs()
    for d in docs:                                               # each document through a fixed-size docs=1 pipeline
        H, W = d["photo_u8"].shape[:2]
        one = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=1, height=H, width=W)
        h1 = {k: d[k].contiguous().pin_memory() for k in KEYS}
        h1["photo_u8"] = d["photo_u8"].unsqueeze(0).contiguous().pin_memory()
        d["fixed"] = one.run_host(h1)[0].clone()
    captures = []
    real_graph = torch.cuda.graph
    monkeypatch.setattr(torch.cuda, "graph", lambda *a, **k: (captures.append(1), real_graph(*a, **k))[1])
    P = sum(H * W for H, W in PIPE_SIZES[:3])
    pipe = DewarpPipeline(model, diffusion_steps=3, n_batch=2, docs=3, max_pixels=P)

    def check(got, batch_docs):
        """byte-equal to dewarp_fullres with the pipeline's map; <= 1 LSB of a fixed-size docs=1 pipeline"""
        assert len(got) == len(batch_docs)
        for i, (g, d) in enumerate(zip(got, batch_docs)):
            ph = d["photo_u8"].to(dev)
            assert torch.equal(g.to(dev), dewarp_fullres(pipe.map64[i:i + 1], ph.unsqueeze(0))[0])
            diff = (g.cpu().int() - d["fixed"].int()).abs()
            assert int(diff.max()) <= 1 and float((diff != 0).float().mean()) < 0.01

    # synchronous host calls, then short batches of 1, 3 and 2 documents
    full = docs[:3]
    check([g.clone() for g in pipe.run_host(_batch(full))], full)
    for sel in ([3], [0, 1, 2], [2, 3]):
        batch = [docs[i] for i in sel]
        check([g.clone() for g in pipe.run_host(_batch(batch))], batch)
    n_caps = len(captures)
    assert n_caps == 4                                           # per slot: one sampling graph, one unwarp graph

    # two batches outstanding == the synchronous call
    batches = [[docs[0], docs[1], docs[2]], [docs[3]], [docs[2], docs[0]], [docs[1], docs[3], docs[0]]]
    tickets, outs = [], []
    for i, b in enumerate(batches):
        tickets.append(pipe.submit_host(_batch(b)))
        if i >= 1:
            outs.append([g.clone() for g in pipe.wait(tickets[i - 1])])
    outs.append([g.clone() for g in pipe.wait(tickets[-1])])
    assert len(captures) == n_caps                               # every composition replays the slot's graphs
    for got, b in zip(outs, batches):
        want = pipe.run_host(_batch(b))
        assert all(torch.equal(x, y) for x, y in zip(got, want))

    # device-resident inputs: the photos are read in place
    dset = {k: v.to(dev) for k, v in _batch(full).items() if k != "photo_u8"}
    dset["photo_u8"] = [d["photo_u8"].to(dev) for d in full]
    for _ in range(2):
        got = [g.clone() for g in pipe.run_device(dset)]
        check(got, full)
    dset["photo_u8"] = [docs[3]["photo_u8"].to(dev), docs[0]["photo_u8"].to(dev), docs[1]["photo_u8"].to(dev)]
    n_caps = len(captures)
    got = pipe.run_device(dset)
    assert len(captures) == n_caps
    for i, g in enumerate(got):
        assert torch.equal(g, dewarp_fullres(pipe.map64[i:i + 1], dset["photo_u8"][i].unsqueeze(0))[0])

    # input from outside
    big = torch.zeros((P // 100 + 1, 100, 3), dtype=torch.uint8)
    bad = [[big], [docs[0]["photo_u8"].float()], [docs[0]["photo_u8"].transpose(0, 1)], [docs[0]["photo_u8"][..., :2].contiguous()],
           [docs[0]["photo_u8"].to(dev)], [], [docs[0]["photo_u8"]] * 4, [docs[0]["photo_u8"].reshape(-1)]]
    for photos in bad:
        h = _batch([docs[0]] * max(1, min(len(photos), 3)))
        h["photo_u8"] = photos
        with pytest.raises(ValueError):
            pipe.submit_host(h)
    with pytest.raises(ValueError):
        pipe.run_device(dict(dset, photo_u8=dset["photo_u8"][:2]))
