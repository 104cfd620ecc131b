"""The denoiser's 512x512 input computed from the photo on the GPU: the numpy oracle (oracle/resize512.py) against cv2.resize, the
host-only planner dvd_y512_u8_plan and the C layout without a GPU; on the GPU, photo_to_y512 and DewarpPipeline(y512_from_photo=True)
against the oracle, byte for byte."""
import ctypes as C
import os
import subprocess

import cv2
import numpy as np
import pytest
import torch

from oracle import synth
from oracle.resize512 import resize512_u8, y512_from_photo

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))

SIZES = [(1500, 2000), (2000, 1500), (4032, 3024), (3000, 4000), (1333, 999), (777, 1333), (1024, 1024), (1024, 2048), (2048, 2048),
         (1023, 1025), (513, 511), (512, 512), (300, 400), (256, 1024), (1, 1), (2, 3), (1, 640)]
# thin photos 1xN and Nx1: every N up to 200, every 7th up to 4096, and the phone sizes
THIN_N = sorted(set(range(1, 200)) | set(range(200, 4097, 7)) | {3000, 3024, 4000, 4032, 6000, 8064})


def _cv2(p: np.ndarray) -> np.ndarray:
    return cv2.resize(p, (512, 512), interpolation=cv2.INTER_LINEAR)


def _random(H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def _page(H, W, seed):
    return synth.make_photo(H, W, seed, "page")[0].permute(1, 2, 0).to(torch.uint8).numpy().copy()


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("H,W", SIZES)
def test_oracle_equals_cv2_resize(H, W):
    for p in (_random(H, W, H * 7 + W), _page(H, W, H + W)):
        assert np.array_equal(resize512_u8(p), _cv2(p))


def test_oracle_equals_cv2_resize_on_thin_photos():
    rng = np.random.default_rng(5)
    for n in THIN_N:
        for shape in ((1, n, 3), (n, 1, 3)):
            p = rng.integers(0, 256, shape, dtype=np.uint8)
            assert np.array_equal(resize512_u8(p), _cv2(p)), shape


def test_oracle_y512_is_the_loaders_float_image():
    for H, W in [(1500, 2000), (3, 700), (512, 512)]:
        p = _random(H, W, 11)
        want = torch.from_numpy(_cv2(p)).permute(2, 0, 1).float() / 255
        got = torch.from_numpy(y512_from_photo(p))
        assert got.dtype == torch.float32 and got.shape == (3, 512, 512) and torch.equal(got, want)
    # an IEEE division: x / 255 and x * (1 / 255) differ on many byte values, the oracle follows the division
    v = np.arange(256, dtype=np.float32)
    assert np.sum(v / np.float32(255) != v * np.float32(1 / 255)) > 100


def _plan(docs, table_bytes=None):
    """docs: (photo pointer, H, W) tuples -> (rc, error message, table bytes)"""
    from dvd_b200 import _lib
    l = _lib.lib()
    n = len(docs)
    arr = (_lib.Y512Doc * max(n, 1))(*[_lib.Y512Doc(p, H, W) for p, H, W in docs])
    nb = l.dvd_y512_table_bytes(n) if table_bytes is None else table_bytes
    table = C.create_string_buffer(max(nb, 1))
    rc = l.dvd_y512_u8_plan(arr if n else None, n, table, nb)
    return rc, l.dvd_last_error().decode(), table.raw


def test_plan_without_a_gpu():
    from dvd_b200 import _lib
    l = _lib.lib()
    assert l.dvd_y512_table_bytes(0) == 16 and l.dvd_y512_table_bytes(16) == 16 + 16 * 32
    rc, msg, _ = _plan([(0x1000, 4032, 3024), (0x2000, 1, 1), (0x3000, 1, 8064)])
    assert rc == 0, msg
    rc, msg, raw = _plan([])                                      # n = 0 plans an empty batch
    assert rc == 0 and raw[:4] == b"\0\0\0\0", msg


PLAN_ERRORS = {  # case -> (docs, table bytes or None, message)
    "H0": ([(0x1000, 10, 10), (0x1000, 0, 10)], None, "y512_u8_plan: document 1 has size 0x10"),
    "W0": ([(0x1000, 10, 0)], None, "y512_u8_plan: document 0 has size 10x0"),
    "negative": ([(0x1000, -3, 10)], None, "y512_u8_plan: document 0 has size -3x10"),
    "null_photo": ([(0x1000, 10, 10), (0, 10, 10)], None, "y512_u8_plan: document 1 has a null photo pointer"),
    "too_large": ([(0x1000, 32768, 21846)], None, "y512_u8_plan: document 0 (32768x21846x3) is too large"),
    "table": ([(0x1000, 10, 10)] * 2, 16 + 32, "y512_u8_plan: table of 48 bytes is too small for 2 documents"),
}


@pytest.mark.parametrize("case", sorted(PLAN_ERRORS))
def test_plan_rejects_bad_input(case):
    docs, nb, msg = PLAN_ERRORS[case]
    rc, got, _ = _plan(docs, nb)
    assert rc == -1 and got.startswith(msg), got


def test_plan_limit_is_exclusive():
    assert _plan([(0x1000, 32768, 21845)])[0] == 0             # 32768 * 21845 * 3 < 2^31


def test_y512_doc_layout_matches_c(tmp_path):
    from dvd_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvd_b200.h"\nint main(){printf("%zu %zu %zu %zu\\n",'
                   'sizeof(dvd_y512_doc_t),offsetof(dvd_y512_doc_t,photo),offsetof(dvd_y512_doc_t,H),offsetof(dvd_y512_doc_t,W));'
                   'return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = _lib.Y512Doc
    assert got == [C.sizeof(D), D.photo.offset, D.H.offset, D.W.offset]


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dvd_b200 import _lib
    _lib.check(_lib.lib().dvd_check_device(), "dvd_check_device")
    return torch.device("cuda:0")


def _want(p: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(y512_from_photo(p))


@pytest.mark.gpu
def test_photo_to_y512_fixed_batch(dev):
    from dvd_b200.inputs import photo_to_y512
    for H, W in [(1500, 2000), (4032, 3024), (1, 640), (513, 511)]:
        ph = np.stack([_random(H, W, 1), _page(H, W, 2), _random(H, W, 3)])
        got = photo_to_y512(torch.from_numpy(ph).to(dev))
        assert got.shape == (3, 3, 512, 512) and got.dtype == torch.float32
        for i in range(3):
            assert torch.equal(got[i].cpu(), _want(ph[i])), (H, W, i)


@pytest.mark.gpu
def test_photo_to_y512_mixed_list_is_one_launch(dev):
    from dvd_b200 import _lib
    from dvd_b200.inputs import photo_to_y512
    photos = [_random(H, W, 20 + i) if i % 2 else _page(H, W, 20 + i) for i, (H, W) in enumerate(SIZES)]
    dp = [torch.from_numpy(p).to(dev) for p in photos]
    n = len(dp)
    big = torch.full((n + 2, 3, 512, 512), -7.0, device=dev)     # documents past n stay untouched
    l = _lib.lib()
    torch.cuda.synchronize()
    n0 = l.dvd_launch_count(0)
    got = photo_to_y512(dp, out=big[:n])
    assert l.dvd_launch_count(0) - n0 == 1
    assert got.data_ptr() == big.data_ptr()
    for i, p in enumerate(photos):
        assert torch.equal(big[i].cpu(), _want(p)), SIZES[i]
    assert bool((big[n:] == -7.0).all())


@pytest.mark.gpu
def test_photo_to_y512_thin_photos(dev):
    from dvd_b200.inputs import photo_to_y512
    rng = np.random.default_rng(9)
    for shape_of in (lambda n: (1, n, 3), lambda n: (n, 1, 3)):
        for k in range(0, len(THIN_N), 64):                       # batched: 64 photos per launch
            photos = [rng.integers(0, 256, shape_of(n), dtype=np.uint8) for n in THIN_N[k:k + 64]]
            got = photo_to_y512([torch.from_numpy(p).to(dev) for p in photos]).cpu()
            for i, p in enumerate(photos):
                assert torch.equal(got[i], torch.from_numpy(_cv2(p)).permute(2, 0, 1).float() / 255), p.shape


@pytest.mark.gpu
def test_photo_to_y512_rejects_bad_input(dev):
    from dvd_b200.inputs import photo_to_y512
    ok = torch.zeros((2, 8, 8, 3), dtype=torch.uint8, device=dev)
    for bad in (ok.float(), ok[..., :2].contiguous(), ok[0], torch.zeros((2, 8, 8, 4), dtype=torch.uint8, device=dev),
                [ok[0].float()], [ok[0, :, :, :1].contiguous()], [ok[0].transpose(0, 1)], [ok[0, :0]], [], "photo"):
        with pytest.raises(ValueError):
            photo_to_y512(bad)
    with pytest.raises(ValueError):
        photo_to_y512(ok, out=torch.empty((2, 3, 512, 512), device=dev, dtype=torch.float64))
    for cpu in (ok.cpu(), [ok[0].cpu()]):
        with pytest.raises(RuntimeError):
            photo_to_y512(cpu)


# ---- DewarpPipeline(y512_from_photo=True) against the same pipeline fed the oracle's y512 (the pipeline is deterministic)
KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")
PIPE_SIZES = [(96, 128), (64, 200), (120, 90), (72, 72)]


@pytest.fixture(scope="module")
def model(dev, state_dict_live):
    from dvd_b200.model import DiT
    m = DiT(precision="fp32")
    m.load_state_dict(state_dict_live, strict=False)
    return m.to(dev).eval()


def _doc(i, H, W):
    d = synth.make_doc_inputs(i, H=H, W=W)
    d["photo_u8"] = d["photo"][0].permute(1, 2, 0).to(torch.uint8).contiguous()
    d["y512"] = _want(d["photo_u8"].numpy())[None]             # what the reference loader feeds the denoiser
    return d


def _host(docs, with_y512, stack=True):
    h = {k: torch.cat([d[k] for d in docs]).contiguous().pin_memory() for k in KEYS if with_y512 or k != "y512"}
    h["photo_u8"] = (torch.stack([d["photo_u8"] for d in docs]).pin_memory() if stack else [d["photo_u8"].pin_memory() for d in docs])
    return h


def _device(h, dev):
    return {k: ([p.to(dev) for p in v] if isinstance(v, list) else v.to(dev)) for k, v in h.items()}


def _same(a, b):
    if isinstance(a, list):
        return len(a) == len(b) and all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(a, b))
    return torch.equal(a.cpu(), b.cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("out_size", [None, (50, 70)])
def test_pipeline_fixed_size(dev, model, out_size):
    from dvd_b200.pipeline import DewarpPipeline
    H, W = 120, 90
    docs = [_doc(i, H, W) for i in range(4)]
    kw = dict(diffusion_steps=3, n_batch=2, docs=2, height=H, width=W, out_size=out_size)
    ref, pipe = DewarpPipeline(model, **kw), DewarpPipeline(model, y512_from_photo=True, **kw)
    assert pipe.h2d_bytes == ref.h2d_bytes - 2 * 3 * 512 * 512 * 4
    batches = [docs[:2], docs[2:], docs[1:3]]
    want = [ref.run_host(_host(b, True)).clone() for b in batches]
    # synchronous, then two batches outstanding
    for b, w in zip(batches, want):
        assert _same(pipe.run_host(_host(b, False)), w)
    tickets = [pipe.submit_host(_host(batches[0], False)), pipe.submit_host(_host(batches[1], False))]
    got = [pipe.wait(tickets[0]).clone()]
    tickets.append(pipe.submit_host(_host(batches[2], False)))
    got += [pipe.wait(tickets[1]).clone(), pipe.wait(tickets[2]).clone()]
    assert all(_same(g, w) for g, w in zip(got, want))
    # device-resident inputs; the prep launch is counted
    n0 = pipe.kernel_launches
    r0 = ref.kernel_launches
    for b, w in zip(batches, want):
        assert _same(pipe.run_device(_device(_host(b, False), dev)), w)
        ref.run_device(_device(_host(b, True), dev))
    assert pipe.kernel_launches - n0 == ref.kernel_launches - r0 + len(batches)
    # y512 together with y512_from_photo, and a photo that is not uint8
    with pytest.raises(ValueError):
        pipe.run_host(_host(batches[0], True))
    with pytest.raises(ValueError):
        pipe.run_device(_device(_host(batches[0], True), dev))
    d = _device(_host(batches[0], False), dev)
    d["photo_u8"] = d["photo_u8"].float()
    with pytest.raises(ValueError):
        pipe.run_device(d)
    # the pipeline that takes y512 checks its inputs as well: a photo of the wrong size, a misshapen x_T and a one-document input
    # that would broadcast to both documents
    d = _device(_host(batches[0], True), dev)
    for k, bad in (("photo_u8", d["photo_u8"][:, 1:].contiguous()), ("x_T", d["x_T"][:2]), ("x_T", d["x_T"].double())):
        with pytest.raises(ValueError):
            ref.run_device(dict(d, **{k: bad}))
    h = _host(batches[0], True)
    for k in ("photo_u8", "mask_cat"):
        with pytest.raises(ValueError):
            ref.submit_host(dict(h, **{k: h[k][:1]}))


@pytest.mark.gpu
@pytest.mark.parametrize("out_size", [None, (40, 60)])
def test_pipeline_mixed_size(dev, model, out_size):
    from dvd_b200.pipeline import DewarpPipeline
    docs = [_doc(i, H, W) for i, (H, W) in enumerate(PIPE_SIZES)]
    P = sum(H * W for H, W in PIPE_SIZES[:3])
    kw = dict(diffusion_steps=3, n_batch=2, docs=3, max_pixels=P, out_size=out_size)
    ref, pipe = DewarpPipeline(model, **kw), DewarpPipeline(model, y512_from_photo=True, **kw)
    # short batches of 3, 1 and 2 documents, synchronous and two outstanding
    batches = [[docs[0], docs[1], docs[2]], [docs[3]], [docs[2], docs[0]], [docs[1], docs[3], docs[0]]]
    want = [[g.clone() for g in ref.run_host(_host(b, True, stack=False))] for b in batches]
    for b, w in zip(batches, want):
        assert _same(pipe.run_host(_host(b, False, stack=False)), w)
    tickets, got = [], []
    for i, b in enumerate(batches):
        tickets.append(pipe.submit_host(_host(b, False, stack=False)))
        if i >= 1:
            got.append([g.clone() for g in pipe.wait(tickets[i - 1])])
    got.append([g.clone() for g in pipe.wait(tickets[-1])])
    assert all(_same(g, w) for g, w in zip(got, want))
    # device-resident inputs: exactly `docs` photos
    for b in (batches[0], batches[3]):
        w = [g.clone() for g in ref.run_device(_device(_host(b, True, stack=False), dev))]
        assert _same(pipe.run_device(_device(_host(b, False, stack=False), dev)), w)
    with pytest.raises(ValueError):
        pipe.run_host(_host(batches[1], True, stack=False))
    h = _host(batches[1], False, stack=False)
    h["photo_u8"] = [h["photo_u8"][0].float()]
    with pytest.raises(ValueError):
        pipe.run_host(h)


@pytest.mark.gpu
def test_pipeline_eager(dev, model, monkeypatch):
    from dvd_b200.pipeline import DewarpPipeline
    monkeypatch.setenv("DVD_NO_GRAPH", "1")
    H, W = 96, 128
    docs = [_doc(i, H, W) for i in range(2)]
    kw = dict(diffusion_steps=3, n_batch=2, docs=2, height=H, width=W)
    ref, pipe = DewarpPipeline(model, **kw), DewarpPipeline(model, y512_from_photo=True, **kw)
    assert not pipe.use_graph
    want = ref.run_host(_host(docs, True)).clone()
    assert _same(pipe.run_host(_host(docs, False)), want)
    assert _same(pipe.run_device(_device(_host(docs, False), dev)), want)
    mkw = dict(diffusion_steps=3, n_batch=2, docs=2, max_pixels=2 * H * W)
    want = [g.clone() for g in DewarpPipeline(model, **mkw).run_host(_host(docs, True, stack=False))]
    assert _same(DewarpPipeline(model, y512_from_photo=True, **mkw).run_host(_host(docs, False, stack=False)), want)
