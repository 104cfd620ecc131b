"""JPEG decode on the GPU, byte-equal to cv2.imdecode(buf, IMREAD_COLOR)[..., ::-1] (the reference loader's cv2.imread -> RGB).

On the CPU: the oracle (oracle/jpeg_decode.py) against cv2 over a matrix of files, the host-only planner dvd_jpeg_plan (output sizes
after the EXIF orientation, each rejection by its message) and the C layout of dvd_jpeg_doc_t.  On the GPU: decode_jpeg against cv2
on the same matrix plus camera-sized photos, a mixed batch in one call, a batch with a corrupt scan, and
DewarpPipeline(max_jpeg_bytes=...) against the same pipeline fed the cv2-decoded photos.
"""
import ctypes as C
import io
import os
import subprocess

import cv2
import numpy as np
import pytest
import torch
from PIL import Image, ImageFile

from oracle import synth
from oracle.jpeg_decode import decode as oracle_decode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ImageFile.MAXBLOCK = 1 << 24          # Pillow's optimize=True / restart markers need the whole stream in one buffer
SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440}
PIL_SAMPLING = {"444": 0, "422": 1, "420": 2}


def _cv2(buf: bytes) -> np.ndarray:
    return np.ascontiguousarray(cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR)[..., ::-1])


def _random(H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


def _page(H, W, seed):
    return synth.make_photo(H, W, seed)[0].permute(1, 2, 0).to(torch.uint8).contiguous().numpy()


def enc_cv2(rgb, q=90, sampling="420", rst=0):
    params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    if rst:
        params += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(rgb[..., ::-1]), params)
    assert ok
    return buf.tobytes()


def enc_pil(img, **kw):
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", **kw)
    return b.getvalue()


def _exif(orientation, little_endian=False):
    """an APP1 Exif payload whose IFD0 holds the orientation tag (0x0112, SHORT), in Intel or Motorola byte order"""
    bo = "little" if little_endian else "big"
    u16 = lambda v: v.to_bytes(2, bo)
    return (b"Exif\0\0" + (b"II*\0" if little_endian else b"MM\0*") + (8).to_bytes(4, bo) + u16(1)
            + u16(0x0112) + u16(3) + (1).to_bytes(4, bo) + u16(orientation) + b"\0\0" + b"\0\0\0\0")


SIZES = [(1, 1), (1, 23), (23, 1), (7, 9), (8, 8), (15, 17), (16, 16), (17, 33), (300, 400), (333, 641)]


def _matrix():
    """(id, file) pairs: every size x sampling at q90, the qualities, page content, optimized tables, restart intervals, grayscale
    and the eight orientations in both TIFF byte orders"""
    cases = []
    for i, (H, W) in enumerate(SIZES):
        img = _random(H, W, i)
        for s in ("444", "422", "420"):
            cases.append((f"random{H}x{W}-{s}-q90", enc_cv2(img, 90, s)))
        cases.append((f"gray{H}x{W}", enc_pil(img[..., 1], quality=90)))
    for H, W in ((17, 33), (300, 400)):
        img = _random(H, W, 7)
        for s in ("444", "422", "420"):
            for q in (50, 100):
                cases.append((f"random{H}x{W}-{s}-q{q}", enc_cv2(img, q, s)))
    for H, W in ((300, 400), (333, 641)):
        img = _page(H, W, 3)
        for s in ("444", "422", "420"):
            cases.append((f"page{H}x{W}-{s}", enc_cv2(img, 90, s)))
    img = _random(333, 641, 11)
    for s in ("444", "422", "420"):
        cases.append((f"optimize-{s}", enc_pil(img, quality=90, subsampling=PIL_SAMPLING[s], optimize=True)))
        cases.append((f"cv2-rst2-{s}", enc_cv2(img, 90, s, rst=2)))
        cases.append((f"pil-blocks3-{s}", enc_pil(img, quality=75, subsampling=PIL_SAMPLING[s], restart_marker_blocks=3)))
        cases.append((f"pil-rows1-{s}", enc_pil(img, quality=95, subsampling=PIL_SAMPLING[s], restart_marker_rows=1)))
    cases.append(("gray-rst", enc_pil(img[..., 0], quality=90, restart_marker_blocks=5)))
    img = _random(40, 64, 5)
    for o in range(1, 9):
        cases.append((f"orientation{o}", enc_pil(img, quality=90, exif=_exif(o))))
        cases.append((f"orientation{o}-II", enc_pil(img, quality=90, subsampling=1, exif=_exif(o, True))))
    return cases


_CASES = None


def matrix():
    global _CASES
    if _CASES is None:
        _CASES = _matrix()
    return _CASES


@pytest.mark.parametrize("idx", range(len(SIZES) * 4 + 12 + 6 + 12 + 1 + 16))
def test_oracle_equals_cv2(idx):
    name, buf = matrix()[idx]
    want = _cv2(buf)
    got = oracle_decode(buf)
    assert got.shape == want.shape and np.array_equal(got, want), name


def test_matrix_size():
    assert len(matrix()) == len(SIZES) * 4 + 12 + 6 + 12 + 1 + 16


# ---- the planner, without a GPU
def _plan(files, table_bytes=None, ws_bytes=1 << 40, null=False):
    """-> (rc, message, [(H, W)]) of dvd_jpeg_plan over `files` with fake device pointers"""
    from dvd_b200 import _lib
    l = _lib.lib()
    n = len(files)
    keep = [C.create_string_buffer(f, len(f)) for f in files]
    docs = (_lib.JpegDoc * max(n, 1))()
    for i, k in enumerate(keep):
        docs[i].file_host = None if null else C.addressof(k)
        docs[i].bytes = len(files[i])
        docs[i].file, docs[i].out = 0x1000 * (i + 1), 0x100000 * (i + 1)
    nb = l.dvd_jpeg_table_bytes(n) if table_bytes is None else table_bytes
    table = C.create_string_buffer(max(nb, 1))
    hw = (C.c_int32 * max(2 * n, 1))()
    rc = l.dvd_jpeg_plan(docs, n, table, nb, ws_bytes, hw)
    return rc, l.dvd_last_error().decode(), [(hw[2 * i], hw[2 * i + 1]) for i in range(n)]


def test_plan_reports_sizes_after_orientation():
    img = _random(40, 64, 1)
    files = [enc_pil(img, quality=90, exif=_exif(o, o % 2 == 0)) for o in range(1, 9)] + [enc_cv2(_random(1, 23, 2)), enc_pil(img[..., 0])]
    rc, msg, hw = _plan(files)
    assert rc == 0, msg
    assert hw == [(40, 64)] * 4 + [(64, 40)] * 4 + [(1, 23), (40, 64)]
    from dvd_b200.inputs import jpeg_hw
    assert jpeg_hw(files) == hw


def _patched(buf, marker, offset, value):
    """buf with byte `offset` after the first `marker` (0xFF xx) set to value; offset 0 is the marker code itself"""
    i = buf.index(bytes([0xFF, marker]))
    b = bytearray(buf)
    b[i + 1 + offset] = value
    return bytes(b)


def _rejections():
    img = _random(24, 32, 4)
    base = enc_cv2(img, 90, "420")
    return {
        "progressive": (enc_pil(img, quality=90, progressive=True), "progressive JPEG is not supported"),
        "arithmetic": (_patched(base, 0xC0, 0, 0xC9), "arithmetic coding is not supported"),
        "12-bit": (_patched(base, 0xC0, 3, 12), "12-bit samples are not supported (8-bit only)"),
        "lossless": (_patched(base, 0xC0, 0, 0xC3), "lossless JPEG is not supported"),
        "cmyk": (_cmyk(img), "4 components (CMYK / 4 components) are not supported (1 or 3 only)"),
        "440": (enc_cv2(img, 90, "440"), "sampling 1x2,1x1,1x1 is not supported (4:4:4, 4:2:2 and 4:2:0 only)"),
        "truncated": (base[:len(base) // 2], "missing EOI marker at the end of the file (truncated file?)"),
        "height0": (_height0(base), "height 0 (DNL) is not supported"),
        "adobe-rgb": (_adobe(base, 0), "Adobe transform 0 (RGB-coded) is not supported"),
        "two-scans": (_patched(base, 0xDA, 3, 1), "more than one scan (the first has 1 of 3 components)"),
        "undefined-table": (_patched(base, 0xDA, 5, 0x33), "scan references an undefined Huffman table"),
        "oversubscribed": (_oversubscribed(base), "over-subscribed Huffman table"),
    }


def _cmyk(img):
    b = io.BytesIO()
    Image.fromarray(img).convert("CMYK").save(b, "JPEG", quality=90)
    return b.getvalue()


def _height0(buf):
    i = buf.index(b"\xff\xc0")
    b = bytearray(buf)
    b[i + 5] = b[i + 6] = 0
    return bytes(b)


def _adobe(buf, transform):
    """buf with its JFIF APP0 replaced by an Adobe APP14 of `transform` (JFIF would take precedence)"""
    assert buf[2:4] == b"\xff\xe0"
    seg = b"Adobe" + bytes([0, 100, 0, 0, 0, 0, transform])
    return buf[:2] + b"\xff\xee" + (len(seg) + 2).to_bytes(2, "big") + seg + buf[4 + int.from_bytes(buf[4:6], "big"):]


def _oversubscribed(buf):
    """the first Huffman table with two more 1-bit codes (which take the whole code space) and as many fewer long ones"""
    i = buf.index(b"\xff\xc4")
    b = bytearray(buf)
    left = 2
    for k in range(15, 0, -1):
        take = min(b[i + 5 + k], left)
        b[i + 5 + k] -= take
        left -= take
    b[i + 5] += 2
    return bytes(b)


REJECTIONS = ["progressive", "arithmetic", "12-bit", "lossless", "cmyk", "440", "truncated", "height0", "adobe-rgb", "two-scans",
              "undefined-table", "oversubscribed"]


@pytest.mark.parametrize("case", REJECTIONS)
def test_plan_rejects_unsupported_files(case):
    buf, msg = _rejections()[case]
    good = enc_cv2(_random(8, 8, 0))
    rc, got, _ = _plan([good, buf])
    assert rc == -1 and got == f"jpeg_plan: document 1: {msg}", got
    from dvd_b200.inputs import jpeg_hw
    with pytest.raises(ValueError, match="document 1"):
        jpeg_hw([good, buf])


def test_plan_rejects_bad_arguments():
    good = enc_cv2(_random(8, 8, 0))
    from dvd_b200 import _lib
    need = _lib.lib().dvd_jpeg_table_bytes(2)
    rc, msg, _ = _plan([good, good], table_bytes=need - 1)
    assert rc == -1 and msg.startswith(f"jpeg_plan: table of {need - 1} bytes is too small for 2 documents"), msg
    rc, msg, _ = _plan([good], null=True)
    assert rc == -1 and msg == "jpeg_plan: document 0: null file pointer or empty file", msg
    rc, msg, _ = _plan([good], ws_bytes=1000)
    assert rc == -1 and msg.startswith("jpeg_plan: the batch needs more than the workspace's 1000 bytes"), msg
    rc, msg, _ = _plan([good, good], ws_bytes=_lib.lib().dvd_jpeg_workspace_bytes(2, 2 * 64, 2 * len(good)))
    assert rc == 0, msg
    rc, msg, _ = _plan([b"not a jpeg"])
    assert rc == -1 and msg == "jpeg_plan: document 0: not a JPEG file (no SOI marker)", msg


def test_jpeg_doc_layout_matches_c(tmp_path):
    from dvd_b200 import _lib
    src = tmp_path / "layout.c"
    f = ["file_host", "bytes", "file", "out"]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvd_b200.h"\nint main(){printf("%zu'
                   + " %zu" * len(f) + '\\n",sizeof(dvd_jpeg_doc_t)' + "".join(f",offsetof(dvd_jpeg_doc_t,{x})" for x in f)
                   + ');return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = _lib.JpegDoc
    assert got == [C.sizeof(D)] + [getattr(D, x).offset for x in f]


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dvd_b200 import _lib
    _lib.check(_lib.lib().dvd_check_device(), "dvd_check_device")
    return torch.device("cuda:0")


def _equal(name, buf, got):
    want = _cv2(buf)
    g = got.cpu().numpy()
    assert g.shape == want.shape, (name, g.shape, want.shape)
    bad = np.argwhere((g != want).any(-1))
    assert len(bad) == 0, (name, len(bad), bad[:4].tolist())


@pytest.mark.gpu
def test_decode_matrix(dev):
    from dvd_b200.inputs import decode_jpeg
    cases = matrix()
    for name, buf in cases:                                   # one file a call
        _equal(name, buf, decode_jpeg([buf], dev)[0])
    outs = decode_jpeg([b for _, b in cases], dev)            # all in one call
    for (name, buf), o in zip(cases, outs):
        _equal(name, buf, o)


@pytest.fixture(scope="module")
def camera():
    """photos of a camera's sizes: a synthetic page at 4032x3024 and its crops / transposes"""
    page = _page(3024, 4032, 7)
    return {(3024, 4032): page, (4032, 3024): np.ascontiguousarray(page.transpose(1, 0, 2)[:, ::-1]),
            (1500, 2000): np.ascontiguousarray(page[700:2200, 1000:3000])}


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(1500, 2000), (3024, 4032), (4032, 3024)])
@pytest.mark.parametrize("q", [90, 95])
def test_decode_camera_sizes(dev, camera, size, q):
    from dvd_b200.inputs import decode_jpeg
    img = camera[size]
    files = {}
    for s in ("444", "422", "420"):
        files[f"{s}"] = enc_cv2(img, q, s)
        files[f"{s}-rst"] = enc_cv2(img, q, s, rst=8)
    files["pil-rows"] = enc_pil(img, quality=q, subsampling=2, restart_marker_rows=1)
    names = list(files)
    outs = decode_jpeg([files[n] for n in names], dev)
    for n, o in zip(names, outs):
        _equal(f"{size} q{q} {n}", files[n], o)


@pytest.mark.gpu
def test_decode_camera_orientations(dev, camera):
    from dvd_b200.inputs import decode_jpeg
    img = camera[(1500, 2000)]
    files = [enc_pil(img, quality=90, subsampling=2, exif=_exif(o, o > 4)) for o in range(1, 9)]
    for o, (buf, got) in enumerate(zip(files, decode_jpeg(files, dev)), 1):
        _equal(f"orientation {o}", buf, got)


@pytest.mark.gpu
def test_decode_mixed_batch_of_16(dev, camera):
    from dvd_b200.inputs import decode_jpeg
    from dvd_b200 import _lib
    rng = np.random.default_rng(5)
    files = []
    for i in range(16):
        H, W = int(rng.integers(1, 900)), int(rng.integers(1, 900))
        img = _page(H, W, i) if i % 2 else _random(H, W, i)
        s = ("444", "422", "420")[i % 3]
        if i % 5 == 0:
            files.append(enc_pil(img[..., 0], quality=85))
        elif i % 4 == 1:
            files.append(enc_pil(img, quality=90, subsampling=PIL_SAMPLING[s], exif=_exif(5 + i % 4)))
        else:
            files.append(enc_cv2(img, 80 + i, s, rst=i % 3))
    files[7] = enc_cv2(camera[(1500, 2000)], 90, "420")
    n0 = _lib.lib().dvd_launch_count(0)
    outs = decode_jpeg(files, dev)
    assert _lib.lib().dvd_launch_count(0) - n0 == 9                 # the same launches whatever the batch
    for i, (buf, o) in enumerate(zip(files, outs)):
        _equal(f"photo {i}", buf, o)


@pytest.mark.gpu
def test_corrupt_scan_stays_in_its_document(dev, camera):
    from dvd_b200.inputs import decode_jpeg
    files = [enc_cv2(camera[(1500, 2000)], 90, s, rst=r) for s, r in (("420", 0), ("444", 4), ("422", 0), ("420", 0))]
    i = files[1].index(b"\xff\xda")
    start = i + 2 + int.from_bytes(files[1][i + 2:i + 4], "big")
    noise = np.random.default_rng(9).integers(0, 256, len(files[1]) - 2 - start, dtype=np.uint8).tobytes()
    bad = bytearray(files[1])
    bad[start:len(bad) - 2] = noise
    for corrupt in (1, 3):
        batch = list(files)
        batch[corrupt] = bytes(bad)
        outs = decode_jpeg(batch, dev)
        torch.cuda.synchronize()
        assert tuple(outs[corrupt].shape) == (1500, 2000, 3)
        for j, (buf, o) in enumerate(zip(batch, outs)):
            if j != corrupt:
                _equal(f"photo {j} next to corrupt {corrupt}", buf, o)


@pytest.mark.gpu
def test_decode_jpeg_checks_arguments(dev):
    from dvd_b200.inputs import decode_jpeg
    good = enc_cv2(_random(20, 30, 1))
    with pytest.raises(ValueError, match="progressive"):
        decode_jpeg([good, enc_pil(_random(8, 8, 0), progressive=True)], dev)
    with pytest.raises(ValueError):
        decode_jpeg([], dev)
    with pytest.raises(ValueError):
        decode_jpeg([good], dev, out=[torch.empty((30, 20, 3), dtype=torch.uint8, device=dev)])
    out = [torch.empty((20, 30, 3), dtype=torch.uint8, device=dev)]
    assert decode_jpeg([good], dev, out=out)[0] is out[0]
    _equal("out", good, out[0])


# ---- DewarpPipeline(max_jpeg_bytes=...) against the same pipeline fed the cv2-decoded photos
KEYS = ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")


@pytest.fixture(scope="module")
def model(dev, state_dict_live):
    from dvd_b200.model import DiT
    m = DiT(precision="fp32")
    m.load_state_dict(state_dict_live, strict=False)
    return m.to(dev).eval()


def _doc(i, H, W, orientation=1):
    d = synth.make_doc_inputs(i, H=H, W=W)
    photo = d["photo"][0].permute(1, 2, 0).to(torch.uint8).numpy()
    if orientation >= 5:                                    # stored transposed; the EXIF tag turns it back to H x W
        photo = np.ascontiguousarray(photo.transpose(1, 0, 2))
    d["jpeg"] = enc_pil(photo, quality=90, subsampling=i % 3, exif=_exif(orientation))
    d["photo_u8"] = torch.from_numpy(_cv2(d["jpeg"]))
    return d


def _host(docs, with_y512, jpeg, stack=True):
    h = {k: torch.cat([d[k] for d in docs]).contiguous().pin_memory() for k in KEYS if with_y512 or k != "y512"}
    if jpeg:
        h["photo_jpeg"] = [d["jpeg"] for d in docs]
    else:
        h["photo_u8"] = (torch.stack([d["photo_u8"] for d in docs]).pin_memory() if stack else
                         [d["photo_u8"].pin_memory() for d in docs])
    return h


def _same(a, b):
    if isinstance(a, list):
        return len(a) == len(b) and all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(a, b))
    return torch.equal(a.cpu(), b.cpu())


def _run_both(ref, pipe, batches, with_y512, stack):
    """each batch through ref (photo_u8) and pipe (photo_jpeg): run_host twice (graph replay), then submit_host + wait with two
    batches outstanding"""
    clone = lambda r: [g.clone() for g in r] if isinstance(r, list) else r.clone()
    want = [clone(ref.run_host(_host(b, with_y512, False, stack))) for b in batches]
    for _ in range(2):
        for b, w in zip(batches, want):
            assert _same(pipe.run_host(_host(b, with_y512, True)), w)
    tickets, got = [], []
    for i, b in enumerate(batches):
        tickets.append(pipe.submit_host(_host(b, with_y512, True)))
        if i >= 1:
            got.append(clone(pipe.wait(tickets[i - 1])))
    got.append(clone(pipe.wait(tickets[-1])))
    assert all(_same(g, w) for g, w in zip(got, want))


@pytest.mark.gpu
def test_pipeline_fixed_size_jpeg(dev, model):
    from dvd_b200.pipeline import DewarpPipeline
    H, W = 120, 90
    docs = [_doc(i, H, W, orientation=(1, 6, 3, 8)[i]) for i in range(4)]
    kw = dict(diffusion_steps=3, n_batch=2, docs=2, height=H, width=W)
    ref = DewarpPipeline(model, **kw)
    pipe = DewarpPipeline(model, max_jpeg_bytes=max(len(d["jpeg"]) for d in docs), **kw)
    assert pipe.h2d_bytes < ref.h2d_bytes
    _run_both(ref, pipe, [docs[:2], docs[2:], docs[1:3]], True, True)
    # run_device is unchanged: decode_jpeg's output feeds it
    from dvd_b200.inputs import decode_jpeg
    h = _host(docs[:2], True, False)
    want = ref.run_host(h).clone()
    d = {k: v.to(dev) for k, v in h.items() if k != "photo_u8"}
    d["photo_u8"] = torch.stack(decode_jpeg([x["jpeg"] for x in docs[:2]], dev))
    assert _same(pipe.run_device(d), want)
    # wrong count, wrong size, too large, photo_u8 instead of photo_jpeg, a file the decoder does not take
    h = _host(docs[:2], True, True)
    for bad in ([docs[0]["jpeg"]], [docs[0]["jpeg"], enc_cv2(_random(90, 120, 0))],
                [docs[0]["jpeg"], docs[1]["jpeg"] + b"\0" * (pipe.max_jpeg_bytes + 1)],
                [docs[0]["jpeg"], enc_pil(_random(H, W, 0), progressive=True)], "not a list"):
        with pytest.raises(ValueError):
            pipe.run_host(dict(h, photo_jpeg=bad))
    with pytest.raises(ValueError):
        pipe.run_host(dict(h, photo_u8=_host(docs[:2], True, False)["photo_u8"]))


@pytest.mark.gpu
def test_pipeline_mixed_size_jpeg(dev, model):
    from dvd_b200.pipeline import DewarpPipeline
    sizes = [(96, 128), (64, 200), (120, 90), (72, 72)]
    docs = [_doc(i, H, W, orientation=(1, 6, 1, 7)[i]) for i, (H, W) in enumerate(sizes)]
    P = sum(H * W for H, W in sizes[:3])
    kw = dict(diffusion_steps=3, n_batch=2, docs=3, max_pixels=P)
    ref = DewarpPipeline(model, **kw)
    pipe = DewarpPipeline(model, max_jpeg_bytes=max(len(d["jpeg"]) for d in docs), **kw)
    _run_both(ref, pipe, [[docs[0], docs[1], docs[2]], [docs[3]], [docs[2], docs[0]]], True, False)
    h = _host(docs[:3], True, True)
    for bad in ([], h["photo_jpeg"] + [docs[3]["jpeg"]]):
        with pytest.raises(ValueError):
            pipe.run_host(dict(h, photo_jpeg=bad))
    big = _doc(9, 130, 130)
    with pytest.raises(ValueError):                              # more than max_pixels in all
        pipe.run_host(_host([docs[0], docs[1], big], True, True))


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", [False, True])
def test_pipeline_jpeg_with_y512_from_photo_and_out_size(dev, model, mixed):
    from dvd_b200.pipeline import DewarpPipeline
    H, W = 96, 128
    docs = [_doc(i, H, W, orientation=(1, 2, 6)[i % 3]) for i in range(3)]
    kw = dict(diffusion_steps=3, n_batch=2, docs=2, y512_from_photo=True, out_size=(50, 70))
    kw.update(max_pixels=2 * H * W) if mixed else kw.update(height=H, width=W)
    ref = DewarpPipeline(model, **kw)
    pipe = DewarpPipeline(model, max_jpeg_bytes=max(len(d["jpeg"]) for d in docs), **kw)
    _run_both(ref, pipe, [docs[:2], docs[1:]] + ([[docs[2]]] if mixed else []), False, not mixed)
