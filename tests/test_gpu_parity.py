"""GPU parity tests: the CUDA path (through the C-ABI library) against the CPU oracle and the golden
fixtures produced by the unmodified reference.  Run on the B200 box with ``-m gpu``.

Tolerances (north_star): final backward map within 0.05 px mean / 0.5 px max, i.e. 2.48e-5 / 2.48e-4 in
normalised units at the largest named size (4032 px: px = d * (4032-1)/2), and unwarped image PSNR >= 45 dB
at 1500x2000 and 4032x3024.  Both gates are asserted for the two modes that claim them: ``fp32`` (FFMA) and
``bf16x3`` (tensor cores, split-precision operands: the default / benchmarked mode).  The single-pass ``bf16``
mode is the stated reduced-accuracy mode: <= 1.5e-3 mean / 6e-3 max normalised (SURVEY.md §8(d): the
reference itself moves by 9.5e-4 / 2.7e-3 when its GEMM operands are rounded to bf16); its image PSNR is
measured and asserted against that looser bound only (>= 20 dB), it does NOT meet the 45 dB gate.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import dvd_oracle as O
from oracle import synth

pytestmark = pytest.mark.gpu

FP32_MEAN, FP32_MAX = 0.05 / 2015.5, 0.5 / 2015.5
BF16_MEAN, BF16_MAX = 1.5e-3, 6e-3


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dvd_b200 import _lib
    _lib.check(_lib.lib().dvd_check_device(), "dvd_check_device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def models(dev, state_dict_live):
    from dvd_b200.model import DiT
    out = {}
    for prec in ("fp32", "bf16", "bf16x3"):
        m = DiT(precision=prec)
        m.load_state_dict(state_dict_live, strict=False)
        out[prec] = m.to(dev).eval()
    return out


def _diffusion(S=3):
    from dvd_b200.sampler import create_gaussian_diffusion
    return create_gaussian_diffusion(steps=S, noise_schedule="cosine", predict_xstart=True, rescale_timesteps=True,
                                     rescale_learned_sigmas=True, timestep_respacing="")


def _kwargs(inp):
    return {"init_flow": inp["init_flow"], "src_feat": None, "src_64": None, "y512": inp["y512"], "tmode": "stage_1_dit_cross",
            "mask_cat": inp["mask_cat"], "init_feat": inp["init_feat"], "iter": True, "mask_y512": inp["mask_y512"],
            "line_msk": inp["line_msk"]}


def _sample(model, inp, S=3):
    out, final = _diffusion(S).ddim_sample_loop(model, (inp["y512"].shape[0], 2, 64, 64), clip_denoised=False, model_kwargs=_kwargs(inp),
                                                eta=0.0, n_batch=2, time_variant=True, x_T=inp["x_T"])
    torch.cuda.synchronize()
    return out.cpu(), final


def psnr(a, b, peak=255.0):
    mse = float(((a.double() - b.double()) ** 2).mean())
    return 99.0 if mse == 0 else 10 * np.log10(peak * peak / mse)


# ----------------------------------------------------------------------------------------------- unwarp (K11)
UNWARP_CASES = {"sampled_page": None, "smooth_noise": (0, "smooth", 120, 90, 12, "noise"),
                "adversarial_noise": (1, "adversarial", 64, 200, 13, "noise"), "zero_page_1ch": (2, "zero", 77, 131, 14, "page")}


def _unwarp_case(golden_dir, case):
    if case == "sampled_page":
        g3 = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))
        return torch.from_numpy(g3["sample"]), synth.make_photo(96, 128, 11, "page")
    mid, mkind, H, W, seed, pkind = UNWARP_CASES[case]
    photo = synth.make_photo(H, W, seed, pkind)
    if case == "zero_page_1ch":
        photo = photo[:, :1].contiguous()
    return synth.make_map64(mid, mkind), photo


@pytest.mark.parametrize("case", list(UNWARP_CASES))
def test_unwarp_matches_reference_golden(dev, golden_dir, case):
    from dvd_b200 import dewarp_fullres, fullres_grid
    u = np.load(os.path.join(golden_dir, "unwarp.npz"))
    m, photo = _unwarp_case(golden_dir, case)
    H, W = photo.shape[-2:]
    grid = fullres_grid(m.to(dev), H, W).cpu()
    gd = (grid - torch.from_numpy(u[case + "_grid"])).abs()
    # grid error in pixels of the photo
    assert float(gd[:, 0].max()) * (W - 1) / 2 < 2e-3 and float(gd[:, 1].max()) * (H - 1) / 2 < 2e-3
    img = dewarp_fullres(m.to(dev), photo.to(dev)).cpu()
    ref = torch.from_numpy(u[case + "_img"])
    assert psnr(img, ref) >= 60.0, psnr(img, ref)
    u8 = dewarp_fullres(m.to(dev), photo.to(dev), out_uint8=True).cpu().numpy()[0]
    # .astype(uint8) truncates: where the four taps are (nearly) equal integers the fp32 result sits on an integer
    # boundary and the last bit decides, so +-1 LSB flips are expected on flat page regions (never more than 1 LSB)
    assert np.abs(u8.astype(int) - u[case + "_u8"].astype(int)).max() <= 1
    assert (u8 != u[case + "_u8"]).mean() < 0.05
    assert psnr(torch.from_numpy(u8.astype(np.float32)), torch.from_numpy(u[case + "_u8"].astype(np.float32))) >= 45.0
    # uint8-in / uint8-out variant == fp32 variant truncated (photo values are integers)
    pu8 = photo[0].permute(1, 2, 0).to(torch.uint8).unsqueeze(0).contiguous().to(dev)
    u8b = dewarp_fullres(m.to(dev), pu8).cpu().numpy()[0]
    assert np.array_equal(u8b, u8)


@pytest.mark.parametrize("H,W", [(1500, 2000), (4032, 3024)])
def test_unwarp_fullsize_vs_oracle(dev, H, W):
    """BASELINE configs' photo sizes: PSNR >= 45 dB against the oracle chain (EV:300-306 + grid_sample)."""
    from dvd_b200 import dewarp_fullres
    m = synth.make_map64(5, "smooth")
    photo = synth.make_photo(H, W, 21, "page")
    img = dewarp_fullres(m.to(dev), photo.to(dev)).cpu()
    ref = O.unwarp(m, photo)
    assert psnr(img, ref) >= 45.0
    assert float((img - ref).abs().max()) < 1.0


def _rotation_map(deg, zoom=1.0):
    """64x64 displacement field of a rotation about the page centre (+ zoom): sends some taps outside the photo."""
    t = np.deg2rad(deg)
    ys, xs = torch.meshgrid(torch.linspace(0, 1, 64), torch.linspace(0, 1, 64), indexing="ij")
    cx, cy = xs - 0.5, ys - 0.5
    rx = zoom * (np.cos(t) * cx - np.sin(t) * cy) + 0.5
    ry = zoom * (np.sin(t) * cx + np.cos(t) * cy) + 0.5
    return torch.stack([rx - xs, ry - ys])[None].float().contiguous()


@pytest.mark.parametrize("deg,zoom", [(3.0, 1.0), (12.0, 1.0), (-25.0, 1.3), (0.0, 0.5)])
def test_unwarp_staged_and_gather_tiles_agree_with_oracle(dev, deg, zoom):
    """Shared-memory-staged tiles (small rotations), gather tiles (window larger than the staged box) and tiles with taps
    outside the photo (zeros padding through the TMA out-of-bounds fill) all reproduce the oracle; fp32 and uint8 variants."""
    from dvd_b200 import dewarp_fullres
    H, W = 600, 800
    m = _rotation_map(deg, zoom) + 0.3 * synth.make_map64(9, "smooth")
    photo = synth.make_photo(H, W, 31, "noise")
    ref = O.unwarp(m, photo)
    img = dewarp_fullres(m.to(dev), photo.to(dev)).cpu()
    assert float((img - ref).abs().max()) < 0.5 and psnr(img, ref) >= 60.0, psnr(img, ref)
    pu8 = photo[0].permute(1, 2, 0).to(torch.uint8).unsqueeze(0).contiguous().to(dev)
    u8 = dewarp_fullres(m.to(dev), pu8).cpu()
    f32_u8 = dewarp_fullres(m.to(dev), photo.to(dev), out_uint8=True).cpu()
    # uint8 photos run on the gather kernel, fp32 photos on the TMA-staged one: ulp-level coordinate differences -> rare 1-LSB flips
    d8 = (u8.int() - f32_u8.int()).abs()
    assert int(d8.max()) <= 1 and float((d8 != 0).float().mean()) < 0.01
    assert int((u8[0].int() - ref[0].permute(1, 2, 0).clamp(0, 255).int()).abs().max()) <= 1


def test_unwarp_tma_batched_and_single_channel(dev):
    """The persistent TMA-staged kernel walks tiles of several photos (tile -> image decode, per-image maps, plane index of the
    tensor maps) and handles C = 1: a batch equals the single calls bit for bit and matches the oracle."""
    from dvd_b200 import dewarp_fullres
    H, W = 600, 800
    maps = torch.cat([_rotation_map(4.0) + 0.3 * synth.make_map64(11, "smooth"), 0.5 * synth.make_map64(12, "smooth"),
                      _rotation_map(-8.0, 1.1)])
    photos = torch.cat([synth.make_photo(H, W, 40 + i, "noise" if i % 2 else "page") for i in range(3)])
    both = dewarp_fullres(maps.to(dev), photos.to(dev))
    for i in range(3):
        one = dewarp_fullres(maps[i:i + 1].to(dev), photos[i:i + 1].to(dev))
        assert torch.equal(both[i:i + 1], one)
        ref = O.unwarp(maps[i:i + 1], photos[i:i + 1])
        assert psnr(one.cpu(), ref) >= 60.0 and float((one.cpu() - ref).abs().max()) < 0.5
    gray = photos[:, :1].contiguous()
    g = dewarp_fullres(maps.to(dev), gray.to(dev)).cpu()
    assert psnr(g, O.unwarp(maps, gray)) >= 60.0
    g8 = dewarp_fullres(maps.to(dev), gray.to(dev), out_uint8=True).cpu()             # fp32 in, uint8 HWC out through the TMA store
    assert int((g8.int() - O.unwarp(maps, gray).permute(0, 2, 3, 1).clamp(0, 255).int()).abs().max()) <= 1


def test_unwarp_tma_and_gather_kernels_agree(dev):
    """The TMA-staged kernel (default for fp32 photos, DVD_UNWARP_TMA_U8=1 for uint8 photos) and the global-gather kernel
    (DVD_UNWARP_NO_TMA=1) give the same image up to ulp-level coordinate differences."""
    import subprocess, sys, tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, torch, numpy as np; sys.path.insert(0, %r); from oracle import synth; from dvd_b200 import dewarp_fullres\n"
            "m = synth.make_map64(5, 'smooth', amp=0.02).cuda(); p = synth.make_photo(1500, 2000, 21, 'page').cuda()\n"
            "pu8 = p[0].permute(1, 2, 0).to(torch.uint8).unsqueeze(0).contiguous()\n"
            "np.savez(sys.argv[1], f32=dewarp_fullres(m, p).cpu().numpy(), u8=dewarp_fullres(m, pu8).cpu().numpy(),"
            " mixed=dewarp_fullres(m, p, out_uint8=True).cpu().numpy())\n" % root)
    outs = []
    with tempfile.TemporaryDirectory() as td:
        for k, env in enumerate(({"DVD_UNWARP_NO_TMA": "1"}, {"DVD_UNWARP_TMA_U8": "1"})):
            f = os.path.join(td, "o%d.npz" % k)
            subprocess.run([sys.executable, "-c", code, f], check=True, env=dict(os.environ, **env), timeout=600)
            outs.append(dict(np.load(f)))
    d = np.abs(outs[0]["f32"] - outs[1]["f32"])
    assert float(d.max()) < 0.25 and float(d.mean()) < 1e-3       # ulp-level coordinate differences x sharp page edges
    for key in ("u8", "mixed"):
        d8 = np.abs(outs[0][key].astype(int) - outs[1][key].astype(int))
        assert int(d8.max()) <= 1 and float((d8 != 0).mean()) < 0.01, key


def test_unwarp_properties_and_edges(dev):
    from dvd_b200 import dewarp_fullres, register_model2
    # linearity in the photo: unwarp(a*p1 + p2) == a*unwarp(p1) + unwarp(p2)
    m = synth.make_map64(7, "smooth").to(dev)
    p1, p2 = synth.make_photo(300, 500, 1, "noise").to(dev), synth.make_photo(300, 500, 2, "page").to(dev)
    lhs = dewarp_fullres(m, 0.5 * p1 + p2)
    rhs = 0.5 * dewarp_fullres(m, p1) + dewarp_fullres(m, p2)
    assert float((lhs - rhs).abs().max()) < 1e-3
    # constant photo: inside pixels stay constant, zero padding only lowers values
    const = torch.full((1, 3, 200, 300), 200.0, device=dev)
    o = dewarp_fullres(torch.zeros(1, 2, 64, 64, device=dev), const)
    assert float(o.max()) <= 200.0 + 1e-3 and float(o[:, :, 5:-5, 5:-5].min()) >= 200.0 - 1e-3
    # batch of photos == one at a time; ragged sizes (W not a multiple of 4, single row / column)
    for (H, W) in [(33, 61), (1, 17), (19, 1), (2, 2)]:
        ph = synth.make_photo(H, W, 3, "noise")
        mm = synth.make_map64(3, "adversarial")
        got = dewarp_fullres(mm.to(dev), ph.to(dev)).cpu()
        assert psnr(got, O.unwarp(mm, ph)) >= 60.0, (H, W)
    two_m = torch.cat([synth.make_map64(1, "smooth"), synth.make_map64(2, "smooth")]).to(dev)
    two_p = torch.cat([synth.make_photo(64, 96, 4, "noise"), synth.make_photo(64, 96, 5, "noise")]).to(dev)
    both = dewarp_fullres(two_m, two_p)
    for i in range(2):
        assert torch.equal(both[i:i + 1], dewarp_fullres(two_m[i:i + 1], two_p[i:i + 1]))
    # empty batch is a no-op
    assert dewarp_fullres(torch.zeros(0, 2, 64, 64, device=dev), torch.zeros(0, 3, 8, 8, device=dev)).shape[0] == 0
    # reg_model_bilin drop-in (WP:14-23) vs torch grid_sample semantics restated in the oracle
    reg = register_model2((512, 512), "bilinear")
    img = torch.rand(2, 5, 40, 50)
    grid = torch.rand(2, 2, 30, 20) * 2.4 - 1.2
    assert float((reg([img.to(dev), grid.to(dev)]).cpu() - O.grid_sample_ref(img, grid)).abs().max()) < 1e-5


# ----------------------------------------------------------------------------------------------- building blocks
def _run_gemm(dev, M, N, K, prec):
    from dvd_b200 import _lib
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A, W, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    Ad, Wd, bd = A.to(dev), W.to(dev), b.to(dev)
    Cd = torch.empty(M, N, device=dev)
    scratch = torch.empty((M + N) * K * 4 + (64 << 10), dtype=torch.uint8, device=dev)   # 16-bit operands (+ lo halves)
    _lib.check(_lib.lib().dvd_test_gemm(_lib.ptr(Ad), _lib.ptr(Wd), _lib.ptr(bd), _lib.ptr(Cd), M, N, K, prec, _lib.ptr(scratch),
                                        scratch.numel(), _lib.stream_ptr()), "dvd_test_gemm")
    torch.cuda.synchronize()
    return Cd.cpu(), A, W, b


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 384, 1032), (2048, 1536, 384), (384, 64, 36), (130, 72, 100)])
def test_gemm_fp32(dev, M, N, K):
    Cg, A, W, b = _run_gemm(dev, M, N, K, 0)
    ref = (A.double() @ W.double().t() + b.double()).float()
    assert float((Cg - ref).abs().max()) < 2e-4 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 384, 1032), (2048, 1536, 384), (8192, 1152, 384), (2048, 4608, 1536),
                                   (2048, 384, 1536)])
def test_gemm_bf16_tcgen05(dev, M, N, K):
    Cg, A, W, b = _run_gemm(dev, M, N, K, 1)
    ref = (A.bfloat16().double() @ W.bfloat16().double().t() + b.double()).float()     # same operand rounding, exact accumulate
    assert float((Cg - ref).abs().max()) < 2e-3 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 384, 1032), (2048, 1536, 1536), (8192, 1152, 384), (2048, 4608, 1536),
                                   (8192, 384, 1536), (2048, 1536, 2048), (2048, 2048, 1536), (512, 64, 64), (384, 192, 128)])
def test_gemm_bf16x3_tcgen05(dev, M, N, K):
    """Split-precision GEMM (three tcgen05 passes): fp32-accurate.  Covers the persistent CTA-pair kernel on the decoder / DiT shapes,
    every tile width, and the generic single-CTA kernel (M = 128 / 384)."""
    Cg, A, W, b = _run_gemm(dev, M, N, K, 2)
    ref = (A.double() @ W.double().t() + b.double()).float()
    err = float((Cg - ref).abs().max()) / max(1.0, float(ref.abs().max()))
    assert err < 4e-5, err


@pytest.mark.parametrize("M,N,K", [(2048, 4608, 1536), (256, 64, 64), (512, 384, 1032), (2048, 1536, 2048)])
def test_gemm_fp16_activation_x_weight_pair(dev, M, N, K):
    """Two-pass mode of the CTA-pair kernel (the decoder's q|k|v GEMM in bf16x3): ONE fp16 activation operand x weight hi + lo.
    Exact against the fp16-rounded activation times the full weight."""
    Cg, A, W, b = _run_gemm(dev, M, N, K, 3)
    ref = (A.half().double() @ W.double().t() + b.double()).float()
    err = float((Cg - ref).abs().max()) / max(1.0, float(ref.abs().max()))
    assert err < 4e-5, err
    full = (A.double() @ W.double().t() + b.double()).float()                        # and fp16-close to the unrounded product
    assert float((Cg - full).abs().max()) / max(1.0, float(full.abs().max())) < 1e-3


@pytest.mark.parametrize("mode", ["bf16x3", "bf16"])
@pytest.mark.parametrize("M,N,K", [(2048, 2048, 1536), (512, 192, 128), (256, 64, 64)])
def test_gemm_decoder_epilogues(dev, mode, M, N, K):
    """The decoder's epilogue specialisations of the CTA-pair kernel through dvd_gemm_tune: folded BN + ReLU into a bf16 hi/lo pair
    (conv1: 16-byte stores after the quad transpose) and folded BN + ReLU + in-place fp32 residual (conv2), every tile width."""
    from dvd_b200 import _lib
    g = torch.Generator(device=dev).manual_seed(M + N + K)
    A = torch.randn(M, K, device=dev, generator=g) * 0.5
    W = torch.randn(N, K, device=dev, generator=g) / K ** 0.5
    sc, sh = torch.rand(N, device=dev, generator=g) + 0.5, torch.randn(N, device=dev, generator=g)
    Ah, Wh = A.bfloat16(), W.bfloat16()
    x3 = mode == "bf16x3"
    Al = (A - Ah.float()).bfloat16() if x3 else None
    Wl = (W - Wh.float()).bfloat16() if x3 else None
    a64 = (Ah.double() + Al.double()) if x3 else Ah.double()
    w64 = (Wh.double() + Wl.double()) if x3 else Wh.double()
    ref = torch.relu((a64 @ w64.t()) * sc.double() + sh.double())
    lib = _lib.lib()
    hi = torch.full((M, N), float("nan"), device=dev, dtype=torch.bfloat16)
    lo = torch.full((M, N), float("nan"), device=dev, dtype=torch.bfloat16)
    _lib.check(lib.dvd_gemm_tune(_lib.ptr(Ah), _lib.ptr(Al), K, _lib.ptr(Wh), _lib.ptr(Wl), K, None, _lib.ptr(sc), _lib.ptr(sh), 1,
                                 _lib.ptr(hi), _lib.ptr(lo) if x3 else None, None, None, M, N, K, _lib.stream_ptr()), "gemm_tune conv1")
    got = hi.double() + (lo.double() if x3 else 0.0)
    tol = 2e-5 if x3 else 1e-2
    assert float((got - ref).abs().max()) < tol * max(1.0, float(ref.abs().max()))
    res = torch.randn(M, N, device=dev, generator=g)
    want = ref + res.double()
    _lib.check(lib.dvd_gemm_tune(_lib.ptr(Ah), _lib.ptr(Al), K, _lib.ptr(Wh), _lib.ptr(Wl), K, None, _lib.ptr(sc), _lib.ptr(sh), 1,
                                 None, None, _lib.ptr(res), _lib.ptr(res), M, N, K, _lib.stream_ptr()), "gemm_tune conv2")
    torch.cuda.synchronize()
    assert float((res.double() - want).abs().max()) < 2e-5 * max(1.0, float(want.abs().max()))


def test_gemm_bf16_more_row_tiles_than_grid_y(dev):
    """M / 128 > 65535 row tiles (the 512x512 pyramid levels of >= 32 documents in flight): the tile index is folded into
    gridDim.z, with a ragged last z-slice."""
    from dvd_b200 import _lib
    M, N, K = (65536 + 3) * 128, 64, 64
    g = torch.Generator(device=dev).manual_seed(5)
    A = (torch.randn(M, K, device=dev, generator=g) * 0.5).bfloat16()
    W = (torch.randn(N, K, device=dev, generator=g) / K ** 0.5).bfloat16()
    b = torch.randn(N, device=dev, generator=g)
    out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    _lib.check(_lib.lib().dvd_gemm_bf16(_lib.ptr(A), None, K, _lib.ptr(W), None, K, _lib.ptr(b), _lib.ptr(out), None, M, N, K,
                                        _lib.stream_ptr()), "gemm")
    torch.cuda.synchronize()
    for r0 in (0, 32768 * 128 - 64, 65535 * 128 - 64, 65536 * 128 - 64, M - 256):      # start, z-slice boundaries, ragged tail
        ref = A[r0:r0 + 256].float() @ W.float().t() + b
        assert float((out[r0:r0 + 256].float() - ref).abs().max()) < 3e-2 * max(1.0, float(ref.abs().max())), r0


def _run_attn(dev, B, H, T, d, prec):
    from dvd_b200 import _lib
    g = torch.Generator().manual_seed(B + H + d)
    q, k, v = (torch.randn(B, T, H * d, generator=g) for _ in range(3))
    o = torch.empty(B, T, H * d, device=dev)
    scratch = torch.empty(max(B * H * T * T * 4, B * T * H * d * 12) + 1024, dtype=torch.uint8, device=dev)
    qd, kd, vd = q.to(dev), k.to(dev), v.to(dev)
    _lib.check(_lib.lib().dvd_test_attention(_lib.ptr(qd), _lib.ptr(kd), _lib.ptr(vd), _lib.ptr(o), B, H, T, d, d ** -0.5, prec,
                                             _lib.ptr(scratch), scratch.numel(), _lib.stream_ptr()), "dvd_test_attention")
    torch.cuda.synchronize()
    return o.cpu(), q, k, v


@pytest.mark.parametrize("d", [64, 256])
def test_attention_fp32(dev, d):
    o, q, k, v = _run_attn(dev, 2, 6, 1024, d, 0)
    ref = O._mha_core(q, k, v, 6, d ** -0.5)
    assert float((o - ref).abs().max()) < 2e-5


@pytest.mark.parametrize("d", [64, 256])
def test_attention_bf16_tcgen05(dev, d):
    o, q, k, v = _run_attn(dev, 2, 6, 1024, d, 1)
    ref = O._mha_core(q.bfloat16().float(), k.bfloat16().float(), v.bfloat16().float(), 6, d ** -0.5)
    assert float((o - ref).abs().max()) < 2e-2 and float((o - ref).abs().mean()) < 2e-3


@pytest.mark.parametrize("d", [64, 256])
def test_attention_fp16_tcgen05(dev, d):
    """bf16x3 mode: fp16 Q / K / V^T / P on tcgen05, output as a bf16 hi + lo pair."""
    o, q, k, v = _run_attn(dev, 2, 6, 1024, d, 2)
    ref = O._mha_core(q.half().float(), k.half().float(), v.half().float(), 6, d ** -0.5)
    assert float((o - ref).abs().max()) < 3e-3 and float((o - ref).abs().mean()) < 2.5e-4


def test_attention_d256_single_cta_fallback(dev, monkeypatch):
    """DVD_ATTN_V1=1: the decoder attention on the single-CTA kernel (the path for T not a multiple of 256) gives the same result
    as the CTA-pair kernel to fp16 accuracy."""
    o_pair, q, k, v = _run_attn(dev, 2, 6, 1024, 256, 2)
    monkeypatch.setenv("DVD_ATTN_V1", "1")
    o_v1, _, _, _ = _run_attn(dev, 2, 6, 1024, 256, 2)
    ref = O._mha_core(q.half().float(), k.half().float(), v.half().float(), 6, 256 ** -0.5)
    assert float((o_v1 - ref).abs().max()) < 3e-3 and float((o_pair - o_v1).abs().max()) < 3e-3


# ----------------------------------------------------------------------------------------------- denoiser stages
def test_static_forward_and_first_step_fp32(dev, models, state_dict_live, golden_dir):
    sd, model = state_dict_live, models["fp32"]
    inp = synth.make_doc_inputs(0, H=96, W=128)
    st = np.load(os.path.join(golden_dir, "stages_doc0_step0.npz"))
    g3 = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))
    eng = model.engine(1, 2)
    g = lambda k: inp[k].to(dev).contiguous()
    eng.static_forward(g("y512"), g("mask_cat"), g("mask_y512"), g("line_msk"))
    feat = eng.feat_nhwc().permute(0, 3, 1, 2).cpu()
    np.testing.assert_allclose(feat[:, ::16, ::4, ::4].numpy(), g3["feat_sub"][:1], atol=5e-5, rtol=1e-4)
    pos = sd["noised_obs_pos_embed"]
    for name, key in (("cond", "c_embed"), ("msk6", "m_embed"), ("msk_line", "l_embed")):
        got = eng.tensor(name).view(1, 1024, 384).cpu() - pos
        np.testing.assert_allclose(got[:, ::8, ::8].numpy(), st[key][:1], atol=1e-4, rtol=1e-4)
    tab = eng.tables([2.0])
    np.testing.assert_allclose(tab[0, :384].cpu().numpy(), st["t_emb"][0], atol=2e-6)
    pred = torch.empty(2, 2, 64, 64, device=dev)
    eng.denoise_step(inp["x_T"].to(dev), torch.zeros(2, 2, 64, 64, device=dev), None, True, tab[0], 1.0, 0.0, pred, None)
    torch.cuda.synchronize()
    np.testing.assert_allclose((eng.tensor("r").view(2, 1024, 384).cpu() - pos)[:, ::8, ::8].numpy(), st["r_embed"], atol=1e-4, rtol=1e-4)
    np.testing.assert_allclose((eng.tensor("xe").view(2, 1024, 384).cpu() - pos)[:, ::8, ::8].numpy(), st["obs_embed"], atol=1e-5, rtol=1e-4)
    assert float((pred.cpu() - torch.from_numpy(g3["pred"][0])).abs().max()) < 1e-4


STAGE_TOL = {"fp32": 1e-4, "bf16x3": 2e-4, "bf16": 6e-2}      # max abs error against the reference's stage outputs (values are O(1..10))


@pytest.mark.parametrize("prec", ["fp32", "bf16x3", "bf16"])
def test_block11_and_decoder_stages_match_reference(dev, models, state_dict_live, golden_dir, prec):
    """Stage-level outputs of the first denoiser forward against hooks on the UNMODIFIED reference (oracle/make_golden.py):
    DiT block 11 (x4,x3,x2,x1), adaptive positional encoding, decoder layer 0 and the decoder output (after decoder.layer_norm)."""
    import torch.nn.functional as F
    from dvd_b200 import _lib
    sd, model = state_dict_live, models[prec]
    inp = synth.make_doc_inputs(0, H=96, W=128)
    st = np.load(os.path.join(golden_dir, "stages_doc0_step0.npz"))
    eng = model.engine(1, 2)
    g = lambda k: inp[k].to(dev).contiguous()
    eng.static_forward(g("y512"), g("mask_cat"), g("mask_y512"), g("line_msk"))
    tab = eng.tables([2.0])
    pred = torch.empty(2, 2, 64, 64, device=dev)
    tol = STAGE_TOL[prec]

    def run(stage):
        _lib.lib().dvd_debug_stop_after(stage)
        try:
            eng.denoise_step(inp["x_T"].to(dev), torch.zeros(2, 2, 64, 64, device=dev), None, True, tab[0], 1.0, 0.0, pred, None)
            torch.cuda.synchronize()
        finally:
            _lib.lib().dvd_debug_stop_after(0)
        return eng.tensor("X").view(2, 1024, 1536).cpu().clone()

    def check(got, want, what):
        err = float(np.abs(got - want).max())
        assert err < tol, (what, err)

    X = run(1)                                                     # x1 | x2 | x3 | x4 along the channels (cross_model.py:623)
    blk = np.stack([X[:, ::8, (3 - j) * 384:(4 - j) * 384:8].numpy() for j in range(4)])      # golden order x4, x3, x2, x1
    check(blk, st["block11"], "block11")
    X = run(2)
    check(X.transpose(1, 2).reshape(2, 1536, 32, 32)[:, ::16, ::4, ::4].numpy(), st["posenc"], "posenc")
    X = run(3)
    check(X[:, ::8, ::16].numpy(), st["dec_layer0"], "dec_layer0")
    X = run(8)                                                     # after decoder layer 5
    dec = F.layer_norm(X, (1536,), sd["decoder.layer_norm.weight"], sd["decoder.layer_norm.bias"], 1e-5)
    check(dec[:, ::8, ::16].numpy(), st["decoder"], "decoder")


def test_dropin_model_call_matches_reference(dev, models, golden_dir):
    """model(x, t, **kwargs) with the reference's kwargs (cross_model.py:568-570), second step (explicit init_feat)."""
    g3 = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))
    inp = synth.make_doc_inputs(0, H=96, W=128)
    rep = lambda v: v.repeat(2, 1, 1, 1).to(dev)
    x = torch.from_numpy(g3["x"][0]).to(dev)
    out, feat = models["fp32"](x, torch.tensor([2, 2], device=dev).float() * (1000.0 / 3), init_flow=rep(inp["init_flow"]),
                               init_feat=rep(inp["init_feat"]), y512=rep(inp["y512"]), mask_cat=rep(inp["mask_cat"]),
                               mask_y512=rep(inp["mask_y512"]), line_msk=rep(inp["line_msk"]), tmode="stage_1_dit_cross", iter=True, tv=True)
    assert tuple(out.shape) == (2, 2, 64, 64) and tuple(feat.shape) == (2, 256, 64, 64)
    assert float((out.cpu() - torch.from_numpy(g3["pred"][0])).abs().max()) < 1e-4
    np.testing.assert_allclose(feat.cpu()[:, ::16, ::4, ::4].numpy(), g3["feat_sub"], atol=5e-5, rtol=1e-4)


# ----------------------------------------------------------------------------------------------- end to end
@pytest.mark.parametrize("doc", [0, 1])
def test_sampling_fp32_matches_reference_golden(dev, models, golden_dir, doc):
    g = np.load(os.path.join(golden_dir, f"sample_S3_doc{doc}.npz"))
    out, final = _sample(models["fp32"], synth.make_doc_inputs(doc, H=96, W=128))
    d = (out - torch.from_numpy(g["sample"])).abs()
    assert float(d.mean()) < FP32_MEAN and float(d.max()) < FP32_MAX, (float(d.mean()) * 2015.5, float(d.max()) * 2015.5)
    assert tuple(final["feat_dict"].shape) == (1, 256, 64, 64) and final["sample"] is final["pred_xstart"]


@pytest.mark.parametrize("doc", [0, 1])
def test_sampling_bf16x3_meets_the_fp32_gate(dev, models, golden_dir, doc):
    """The default tensor-core mode (split-precision GEMMs, fp16 attention) is held to the SAME map gate as fp32."""
    g = np.load(os.path.join(golden_dir, f"sample_S3_doc{doc}.npz"))
    out, _ = _sample(models["bf16x3"], synth.make_doc_inputs(doc, H=96, W=128))
    d = (out - torch.from_numpy(g["sample"])).abs()
    assert float(d.mean()) < FP32_MEAN and float(d.max()) < FP32_MAX, (float(d.mean()) * 2015.5, float(d.max()) * 2015.5)


def test_sampling_S10_thresholds_bf16x3(dev, models, golden_dir):
    g = np.load(os.path.join(golden_dir, "sample_S10_doc2.npz"))
    out, _ = _sample(models["bf16x3"], synth.make_doc_inputs(2, H=96, W=128), S=10)
    assert float((out - torch.from_numpy(g["sample"])).abs().max()) < 2e-3


@pytest.mark.parametrize("doc", [0, 1])
def test_sampling_bf16_within_stated_bound(dev, models, golden_dir, doc):
    g = np.load(os.path.join(golden_dir, f"sample_S3_doc{doc}.npz"))
    out, _ = _sample(models["bf16"], synth.make_doc_inputs(doc, H=96, W=128))
    d = (out - torch.from_numpy(g["sample"])).abs()
    assert float(d.mean()) < BF16_MEAN and float(d.max()) < BF16_MAX, (float(d.mean()), float(d.max()))


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_training_rollout_matches_reference_golden(dev, models, golden_dir, prec):
    """SURVEY §8(f) row 4: ddim_sample_loop_for_training (gaussian_diffusion.py:647-780; raw timestep embedding, steps S-1 .. timestep+1,
    one sample) against the unmodified reference's output."""
    g = np.load(os.path.join(golden_dir, "rollout_doc0_t0.npz"))
    inp = synth.make_doc_inputs(0, H=96, W=128)
    kw = {k: inp[k] for k in ("init_flow", "y512", "mask_cat", "init_feat", "mask_y512", "line_msk")}
    out, feat = _diffusion().ddim_sample_loop_for_training(models[prec], (1, 2, 64, 64), noise=None, clip_denoised=False, model_kwargs=kw,
                                                            eta=0.0, progress=True, n_batch=1, time_variant=True, iter=True, mode="train",
                                                            timestep=0, x_T=inp["x_T"][:1])
    torch.cuda.synchronize()
    d = (out.cpu() - torch.from_numpy(g["pred"])).abs()
    assert float(d.mean()) < FP32_MEAN and float(d.max()) < FP32_MAX, (float(d.mean()), float(d.max()))
    np.testing.assert_allclose(feat.cpu()[:, ::16, ::4, ::4].numpy(), g["feat_sub"], atol=2e-4, rtol=1e-3)


def test_sampling_S10_thresholds_fp32(dev, models, golden_dir):
    """S = 10 hits t = 600.0 and 300.0 exactly (strict thresholds of cross_model.py:576-579)."""
    g = np.load(os.path.join(golden_dir, "sample_S10_doc2.npz"))
    out, _ = _sample(models["fp32"], synth.make_doc_inputs(2, H=96, W=128), S=10)
    assert float((out - torch.from_numpy(g["sample"])).abs().max()) < 2e-3


@pytest.mark.parametrize("docs", [3, 17])
@pytest.mark.parametrize("prec", ["fp32", "bf16", "bf16x3"])
def test_document_batch_equals_single_documents(dev, models, prec, docs):
    """Documents are independent: a batch of documents gives the same maps as separate calls.  17 documents are 34 samples, more
    than the 32 of one fp32 attention chunk: the cross attention's second chunk reads K / V from document 16 (kv_div = 2), and the
    self-attention (136 samples) runs in five chunks."""
    inps = [synth.make_doc_inputs(d, with_photo=False) for d in ((0, 1, 5) if docs == 3 else range(docs))]
    cat = {k: torch.cat([i[k] for i in inps]) for k in inps[0]}
    both, _ = _sample(models[prec], cat)
    for j, i in enumerate(inps):
        one, _ = _sample(models[prec], i)
        assert float((both[j:j + 1] - one).abs().max()) < {"fp32": 1e-5, "bf16x3": 1e-5, "bf16": 1e-3}[prec]


def test_pipeline_device_host_and_pipelined_submission_agree(dev, models):
    """DewarpPipeline (the call bench.py times): CUDA-graph replay on device-resident inputs, the synchronous host call and the
    double-buffered submit_host / wait form give the same uint8 images, equal to sampler + dewarp_fullres on the same inputs."""
    from dvd_b200 import dewarp_fullres
    from dvd_b200.pipeline import DewarpPipeline
    H, W = 96, 128
    pipe = DewarpPipeline(models["fp32"], diffusion_steps=3, n_batch=2, docs=1, height=H, width=W)
    docs = [synth.make_doc_inputs(d, H=H, W=W) for d in (0, 1, 5, 0)]
    hosts = []
    for d in docs:
        h = {k: d[k].contiguous().pin_memory() for k in ("y512", "mask_cat", "mask_y512", "line_msk", "x_T")}
        h["photo_u8"] = d["photo"].permute(0, 2, 3, 1).to(torch.uint8).contiguous().pin_memory()
        hosts.append(h)
    want = []
    for d, h in zip(docs, hosts):
        m, _ = _sample(models["fp32"], d)
        want.append(dewarp_fullres(m.to(dev), h["photo_u8"].to(dev)).cpu())
    for h, w in zip(hosts, want):                                    # device-resident inputs, graph replay (twice: capture + replay)
        dset = {k: v.to(dev) for k, v in h.items()}
        for _ in range(2):
            got = pipe.run_device(dset).cpu()
            assert int((got.int() - w.int()).abs().max()) <= 1 and float((got != w).float().mean()) < 0.01
    for h, w in zip(hosts, want):                                    # synchronous host call
        assert torch.equal(pipe.run_host(h).clone(), pipe.run_host(h))
        got = pipe.run_host(h)
        assert int((got.int() - w.int()).abs().max()) <= 1 and float((got != w).float().mean()) < 0.01
    tickets, outs = [], []
    for i, h in enumerate(hosts):                                    # two batches outstanding
        tickets.append(pipe.submit_host(h))
        if i >= 1:
            outs.append(pipe.wait(tickets[i - 1]).clone())
    outs.append(pipe.wait(tickets[-1]).clone())
    for got, h in zip(outs, hosts):
        assert torch.equal(got, pipe.run_host(h))


def test_seeded_noise_consumption_matches_reference_order(dev, models):
    """Without x_T the sampler draws randn(shape) then randn(n_batch, ...) like gaussian_diffusion.py:559-569, and leaves the
    generator where the reference leaves it (one unused randn_like(x) per DDIM step, gaussian_diffusion.py:479), so that the NEXT
    document of a seeded run sees the same noise too."""
    inp = synth.make_doc_inputs(0, with_photo=False)
    torch.manual_seed(123); torch.cuda.manual_seed(123)
    _ = torch.randn(1, 2, 64, 64, device=dev); xT = torch.randn(2, 2, 64, 64, device=dev)
    for _ in range(3):
        torch.randn_like(xT)
    nxt = torch.randn(8, device=dev)
    torch.manual_seed(123); torch.cuda.manual_seed(123)
    a, _ = _diffusion().ddim_sample_loop(models["fp32"], (1, 2, 64, 64), clip_denoised=False, model_kwargs=_kwargs(inp), eta=0.0,
                                         n_batch=2, time_variant=True)
    assert torch.equal(torch.randn(8, device=dev), nxt)
    b, _ = _diffusion().ddim_sample_loop(models["fp32"], (1, 2, 64, 64), clip_denoised=False, model_kwargs=_kwargs(inp), eta=0.0,
                                         n_batch=2, time_variant=True, x_T=xT)
    assert torch.equal(a, b)


@pytest.mark.parametrize("H,W", [(1500, 2000), (4032, 3024)])
@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_end_to_end_dewarp_psnr(dev, models, golden_dir, prec, H, W):
    """Sampling + unwarp of a full-size photo vs the oracle's unwarp of the reference's golden map: PSNR >= 45 dB (north_star),
    for the FFMA mode and for the default tensor-core mode, at both BASELINE photo sizes (fp32 image and truncated uint8)."""
    from dvd_b200 import dewarp_fullres
    g = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))
    inp = synth.make_doc_inputs(0, H=96, W=128)
    out, _ = _sample(models[prec], inp)
    photo = synth.make_photo(H, W, 77, "page")
    img = dewarp_fullres(out.to(dev), photo.to(dev)).cpu()
    ref = O.unwarp(torch.from_numpy(g["sample"]), photo)
    assert psnr(img, ref) >= 45.0, psnr(img, ref)
    img8 = dewarp_fullres(out.to(dev), photo.permute(0, 2, 3, 1).to(torch.uint8).contiguous().to(dev)).cpu()
    ref8 = torch.from_numpy(O.to_uint8_hwc(ref)).unsqueeze(0)
    assert psnr(img8.float(), ref8.float()) >= 45.0, psnr(img8.float(), ref8.float())


def test_bf16_mode_image_error_is_reported_not_gated(dev, models, golden_dir, capsys):
    """Single-pass bf16 is the stated reduced-accuracy mode: its image PSNR at 1500x2000 is measured here (and printed) and only held
    to the looser stated bound; it is below north_star's 45 dB, which is why bf16x3 is the default and benchmarked mode."""
    from dvd_b200 import dewarp_fullres
    g = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))
    out, _ = _sample(models["bf16"], synth.make_doc_inputs(0, H=96, W=128))
    photo = synth.make_photo(1500, 2000, 77, "page")
    p = psnr(dewarp_fullres(out.to(dev), photo.to(dev)).cpu(), O.unwarp(torch.from_numpy(g["sample"]), photo))
    with capsys.disabled():
        print(f"\n[bf16 single-pass] image PSNR at 1500x2000 vs reference map: {p:.1f} dB (gate for fp32 / bf16x3: 45 dB)")
    assert p >= 20.0, p


# ----------------------------------------------------------------------------------------------- kernel variants and the evaluation drop-in
@pytest.mark.parametrize("env", [{"DVD_GEMM_V1": "1"}, {}, {"DVD_GEMM_BN": "256"}, {"DVD_GEMM_BN": "192"}, {"DVD_GEMM_BN": "128"},
                                 {"DVD_GEMM_BN": "64"}])
def test_gemm_kernel_variants_agree(dev, env):
    """The tcgen05 GEMM kernels (generic single-CTA; persistent CTA-pair with every tile width) are selected by
    shape at run time; force each configuration (env is read once per process, hence the subprocess) over the denoiser's shapes in
    both tensor modes."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "gemm_bench.py"), "--check"], env={**os.environ, **env},
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if "relerr" in l]
    assert len(lines) >= 16
    for l in lines:
        assert float(l.split("relerr")[1]) < (1e-2 if " bf16 " in l else 4e-5), l


def test_run_evaluation_docunet_dropin(dev, models, golden_dir, tmp_path, monkeypatch):
    """evaluation.py:142-327 replacement driven with stub preprocessing nets that return the synthetic conditioning tensors:
    the saved PNG equals the oracle's dewarp of the reference's golden map up to the bf16/fp32 tolerance."""
    from PIL import Image
    from dvd_b200.evaluation import run_evaluation_docunet
    inp = synth.make_doc_inputs(0, H=96, W=128)
    g = np.load(os.path.join(golden_dir, "sample_S3_doc0.npz"))

    class Env:
        train_mode = "stage_1_dit_cross"; iter = True; use_gt_mask = False; use_line_mask = True; use_init_flow = False
        clip_denoised = False; n_batch = 2; time_variant = True; visualize = True; eval_dataset_name = "synthetic"

    class Settings:
        env = Env(); name = "t"

    class Dewarp(torch.nn.Module):           # GeoTr_Seg_Inf stand-in: (ref_bm, mask_x)
        def forward(self, x):
            return torch.zeros(1, 2, 288, 288, device=x.device), inp["mask_cat"].to(x.device)

    class Seg(torch.nn.Module):              # U2NETP stand-in: mskx, d0, hx6 .. hx1d (6 x 64 channels @ 64x64 -> 384)
        def forward(self, x):
            parts = inp["mask_y512"].to(x.device).split(64, dim=1)
            return (torch.zeros(1, 3, 288, 288, device=x.device), None) + tuple(parts)

    class Line(torch.nn.Module):
        def forward(self, x):
            return inp["line_msk"].to(x.device), None

    photo = inp["photo"]
    loader = [{"source_image": inp["y512"], "source_image_ori": photo, "path": ["/data/doc0.png"]}]
    monkeypatch.chdir(tmp_path)
    torch.manual_seed(2000)                  # CPU generator: the sampler draws x_T on the model's device, so fix it explicitly below
    diffusion = _diffusion()
    orig = diffusion.ddim_sample_loop
    diffusion.ddim_sample_loop = lambda *a, **k: orig(*a, **{**k, "x_T": inp["x_T"]})
    times = run_evaluation_docunet(Settings, None, loader, diffusion, models["fp32"], Dewarp(), Line(), Seg())
    assert list(times) == [0]
    png = np.asarray(Image.open(tmp_path / "vis_hp" / "synthetic" / "t" / "dewarped_pred" / "warped_doc0.png"))
    ref = O.to_uint8_hwc(O.unwarp(torch.from_numpy(g["sample"]), photo))
    assert png.shape == ref.shape and np.abs(png.astype(int) - ref.astype(int)).max() <= 1
