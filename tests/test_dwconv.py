"""The decoder's depthwise 3x3 convolution + folded BN + ReLU of the tensor modes (dvd_test_dwconv, the launch dvd_denoise_step makes),
against a float64 reference over whole 32x32 token grids: every image border and every boundary between the kernel's row bands is
compared.  Argument validation is checked without a GPU."""
import ctypes as C

import pytest

DVD_E_BADARG = -1


@pytest.fixture(scope="module")
def lib():
    from dvd_b200 import _lib
    return _lib.lib()


def _split(x):
    """x (fp32) -> bf16 hi, bf16 lo with hi + lo exact in fp32"""
    import torch
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return hi, lo


def _inputs(N, Cc, seed, dev):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, 1024, Cc, generator=g)
    u = torch.rand(N, 1024, Cc, generator=g)
    x[u < 0.05] = 0.0                                             # exact zeros
    x[(u >= 0.05) & (u < 0.07)] = -0.0
    x[u > 0.98] *= 3.0e4                                          # large magnitudes, both signs
    hi, lo = _split(x)
    w9 = torch.randn(9, Cc, generator=g) * 0.5
    scale = torch.rand(Cc, generator=g) * 2.0 - 0.5               # includes negative BN scales
    shift = torch.randn(Cc, generator=g) * 0.3
    return [t.to(dev).contiguous() for t in (hi, lo, w9, scale, shift)]


def _reference(v, w9, scale, shift):
    """float64 depthwise 3x3 (zero padding) + BN + ReLU of v [N,1024,C]; also the magnitude sum(|s w v|) + |t| that bounds fp32 rounding"""
    import torch
    N, _, Cc = v.shape
    p = torch.nn.functional.pad(v.double().view(N, 32, 32, Cc), (0, 0, 1, 1, 1, 1))
    acc = torch.zeros(N, 32, 32, Cc, dtype=torch.float64, device=v.device)
    mag = torch.zeros_like(acc)
    for ky in range(3):
        for kx in range(3):
            t = p[:, ky:ky + 32, kx:kx + 32, :] * w9[ky * 3 + kx].double()
            acc += t
            mag += t.abs()
    s, t = scale.double(), shift.double()
    ref = torch.relu(acc * s + t)
    return ref.view(N, 1024, Cc), (mag * s.abs() + t.abs()).view(N, 1024, Cc)


def _run(lib, hi, lo, w9, scale, shift, N, Cc, with_lo=True):
    import torch
    from dvd_b200 import _lib
    out_hi, out_lo = torch.empty_like(hi), torch.empty_like(hi)
    _lib.check(lib.dvd_test_dwconv(_lib.ptr(hi), _lib.ptr(lo) if with_lo else None, _lib.ptr(w9), _lib.ptr(scale), _lib.ptr(shift),
                                   _lib.ptr(out_hi), _lib.ptr(out_lo), N, Cc, _lib.stream_ptr()), "dvd_test_dwconv")
    torch.cuda.synchronize()
    return out_hi, out_lo


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 2, 32])
def test_dwconv_pair_matches_float64(lib, N):
    import torch
    Cc = 2048
    hi, lo, w9, scale, shift = _inputs(N, Cc, 100 + N, torch.device("cuda:0"))
    out_hi, out_lo = _run(lib, hi, lo, w9, scale, shift, N, Cc)
    v = hi.float() + lo.float()                                  # the kernel's fp32 input value
    ref, mag = _reference(v, w9, scale, shift)
    got = out_hi.double() + out_lo.double()
    err = (got - ref).abs()
    tol = 2.0 ** -16 * mag + 1e-6
    bad = err > tol
    assert not bool(bad.any()), f"{int(bad.sum())} outputs off, worst {float((err / tol).max()):.3f} x tolerance"
    assert bool((got >= 0).all())
    assert float((ref > 0).double().mean()) > 0.3                # the ReLU leaves a good share of outputs non-zero


@pytest.mark.gpu
def test_dwconv_single_bf16_input_and_no_lo_output(lib):
    """bf16 mode: in_lo NULL (value = hi alone); out_lo NULL writes the bf16 part only, identical to the pair's hi"""
    import torch
    from dvd_b200 import _lib
    N, Cc = 2, 2048
    hi, lo, w9, scale, shift = _inputs(N, Cc, 7, torch.device("cuda:0"))
    out_hi, _ = _run(lib, hi, lo, w9, scale, shift, N, Cc, with_lo=False)
    ref, mag = _reference(hi.float(), w9, scale, shift)
    err = (out_hi.double() - ref).abs()
    assert bool((err <= 2.0 ** -8 * mag + 1e-6).all())
    only_hi = torch.empty_like(hi)
    _lib.check(lib.dvd_test_dwconv(_lib.ptr(hi), None, _lib.ptr(w9), _lib.ptr(scale), _lib.ptr(shift), _lib.ptr(only_hi), None, N, Cc,
                                   _lib.stream_ptr()), "dvd_test_dwconv")
    torch.cuda.synchronize()
    assert torch.equal(only_hi.view(torch.int16), out_hi.view(torch.int16))


def test_dwconv_rejects_bad_arguments(lib):
    """validation happens before any CUDA call, so it runs without a GPU"""
    p = C.c_void_p(1 << 20)                                       # never dereferenced
    ok = dict(in_hi=p, in_lo=p, w9=p, scale=p, shift=p, out_hi=p, out_lo=p, N=2, C=2048)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.dvd_test_dwconv(a["in_hi"], a["in_lo"], a["w9"], a["scale"], a["shift"], a["out_hi"], a["out_lo"], a["N"], a["C"], None)

    for C_bad in (2048 + 32, 8, 0, -64):
        assert call(C=C_bad) == DVD_E_BADARG, C_bad
        assert b"multiple of 64" in lib.dvd_last_error()
    for N_bad in (0, -1):
        assert call(N=N_bad) == DVD_E_BADARG, N_bad
    for name in ("in_hi", "w9", "scale", "shift", "out_hi"):
        assert call(**{name: None}) == DVD_E_BADARG, name
    assert call(in_hi=C.c_void_p((1 << 20) + 8)) == DVD_E_BADARG     # not 16-byte aligned
    assert call(N=1 << 30) == DVD_E_BADARG                          # more CTAs than one grid dimension holds
