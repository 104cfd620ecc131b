"""The tensor-core attention kernels (k_attn_tc for head dim 64 and, under DVD_ATTN_V1=1, 256; k_attn_pair for 256) through
dvd_test_attention_tc, the launch dvd_denoise_step makes, against float64 softmax on the exact 16-bit operands.

The kernels use a lazy online softmax: the first key tile sets the row maximum m, and a later tile replaces it only when its
maximum exceeds m by more than 8 log2 units (then O in tensor memory and the row sum l are scaled by alpha = 2^(m - m_new)).
Random inputs never grow a row maximum that much, so the designed inputs below are built to reach that branch, and a CPU
shadow of the rule (`shadow_rescales`) asserts that they do, at the intended rows and tiles, under each kernel's tiling
(64 keys per step for k_attn_tc, 128 for k_attn_pair).

Error bound, per element (O the kernel's output, O_ref the float64 result, A = softmax(scale Q K^T) |V|):

    |O - O_ref| <= (2 u_P + T 2^-24 + delta_row) (A + |O_ref|) + u_o |O_ref|

  u_P        rounding of the probabilities P to the operand type: 2^-11 (fp16), 2^-8 (bf16).  P enters the numerator sum_j P_j V_j
             (error <= u_P A relative to the row sum) and, in k_attn_tc and the bf16 pair kernel, the row sum itself (<= u_P |O|);
  T 2^-24    fp32 accumulation of the T-term sums of P V and of l, and ex2.approx (relative error below 2^-22);
  delta_row  error of the fp32 scores in the exponent: 2^-22 scale max_j (|Q| |K|^T)_ij (the inputs keep it below 2^-14);
  u_o        output rounding: 2^-16 for the bf16 hi + lo pair, 2^-8 for bf16 alone.

The fp32 path (dvd_test_attention, precision 0: FFMA GEMM, softmax, FFMA GEMM) gets the same model with fp32 scores:
(2^-20 + 2 T 2^-24 + (d + 2) 2^-23 scale max_j (|Q| |K|^T)_ij) (A + |O_ref|).
"""
import ctypes as C
import math
import re
import zlib
from types import SimpleNamespace

import pytest
import torch

from oracle import dvd_oracle as O

DVD_E_BADARG = -1
LOG2E = 1.0 / math.log(2.0)
THRESHOLD = 8.0              # log2 units of scale * q.k: the stale row maximum is kept while a tile grows it by no more than this
SIG = 9                      # dims 0..8 of q and k carry the designed logits, dims 9..d-1 small noise
SENTINEL = 0x7FC1            # a bf16 NaN pattern no kernel writes: prefilled around and between the output regions

# kernel -> (head dim, DVD_ATTN_V1, keys per step)
KERNELS = {"tc_d64": (64, False, 64), "tc_d256": (256, True, 64), "pair_d256": (256, False, 128)}
CASES = ("ramp", "late_spike", "spike_other_half", "mixed_rows", "threshold_7.5", "threshold_8.5", "near_one_hot", "randn")
RESCALING = {"ramp", "late_spike", "spike_other_half", "mixed_rows", "threshold_8.5", "near_one_hot"}
MIXED_A = (1.0, 0.5, 0.25, 0.0, -0.5)      # per-row slope of the mixed-rows ramp: rescale every tile, every 2nd, every 4th, never


def tile_width(kernel, T):
    """Keys per step of the kernel that runs: attention_tc falls back from the pair to k_attn_tc when T % 256 != 0."""
    d, v1, w = KERNELS[kernel]
    return 64 if w == 128 and T % 256 else w


def shadow_rescales(x2, w):
    """The kernels' lazy-rescale rule replayed on logits x2 [..., T] in log2 units (scale * log2(e) * q.k).

    Returns (rescale [..., T // w] bool: the row's O is rescaled at that key step, peak [...]: the largest exponent of a
    probability, x2 - m, against the maximum m in effect when it is computed)."""
    tm = x2.unflatten(-1, (-1, w)).amax(-1)
    nt = tm.shape[-1]
    out = torch.zeros(tm.shape, dtype=torch.bool)
    m = tm[..., 0].clone()
    peak = tm[..., 0] - m
    for t in range(1, nt):
        grow = (torch.maximum(m, tm[..., t]) - m) > THRESHOLD
        out[..., t] = grow
        m = torch.where(grow, tm[..., t], m)
        peak = torch.maximum(peak, tm[..., t] - m)
    return out, peak


def make_case(case, kernel, T, f16, nsamp=2, heads=2):
    """Designed q, k, v (16-bit, [nsamp, T, heads * d]) and the intended rescales [nsamp, heads, T, T // w] of `case`.

    Logits in log2 units are built from one large coordinate per row and key (q[0] = a_i, k[0] = g_j / (scale log2 e)) plus noise:
      ramp              every step's maximum is 9 above the previous one (a_i in [1, 1.11]): every row rescales at every step
      late_spike        one key in the first half of the last step is 20 above the rest: every row rescales at the last step
      spike_other_half  the same in the second half of the last step (the keys of the partner warp of each row pair)
      mixed_rows        the ramp with a_i = 1, 0.5, 0.25, 0, -0.5 by row: rows of one warp rescale at different steps or never
      threshold_7.5/8.5 a key in the middle grows the maximum by 7.5 (no rescale, P up to 2^7.5) or 8.5 (one rescale)
      near_one_hot      8 row classes (one coordinate each) whose logits span 60, maximum at a random key of the second half
      randn             q, k, v ~ N(0, 1), the suite's usual inputs: no rescale"""
    d = KERNELS[kernel][0]
    w = tile_width(kernel, T)
    nt = T // w
    c = d ** -0.5 * LOG2E
    f64 = torch.float64
    g = torch.Generator().manual_seed(zlib.crc32(f"{case}/{kernel}/{T}".encode()))
    shape = (nsamp, T, heads, d)
    v = torch.randn(shape, generator=g, dtype=f64)
    pos = torch.arange(T)
    steps = torch.arange(nt)
    rows = torch.zeros(T, nt, dtype=torch.bool)                     # intended rescales, the same for every sample and head
    if case == "randn":
        q = torch.randn(shape, generator=g, dtype=f64)
        k = torch.randn(shape, generator=g, dtype=f64)
    else:
        q = torch.zeros(shape, dtype=f64)
        k = torch.zeros(shape, dtype=f64)
        q[..., SIG:] = 0.1 * torch.randn(nsamp, T, heads, d - SIG, generator=g, dtype=f64)
        k[..., SIG:] = 0.1 * torch.randn(nsamp, T, heads, d - SIG, generator=g, dtype=f64)
        if case == "near_one_hot":
            cls = (pos * 5 + pos // 128) % 8                        # classes interleave within every warp
            q[:, pos, :, 1 + cls] = 1.0
            gk = -12.0 - 48.0 * torch.rand(nsamp, heads, T, 8, generator=g, dtype=f64)
            jc = torch.randint(T // 2, T, (nsamp, heads, 1, 8), generator=g)
            gk.scatter_(2, jc, 0.0)
            k[..., 1:9] = (gk / c).permute(0, 2, 1, 3)
            expect = torch.zeros(nsamp, heads, T, nt, dtype=torch.bool)
            expect.scatter_(3, (jc[:, :, 0, :] // w)[:, :, cls].unsqueeze(-1), True)
            return _pack(q, k, v, expect, f16, d, w, heads)
        spread = ((pos * 37) % w).to(f64) / w                       # 0 at the first key of every step
        a = 1.0 + (pos % 8).to(f64) / 64
        if case in ("ramp", "mixed_rows"):
            gk = 9.0 * (pos // w - (nt - 1) / 2) - 3.0 * spread
            if case == "ramp":
                rows[:, 1:] = True
            else:
                a = torch.tensor(MIXED_A, dtype=f64)[pos % len(MIXED_A)]
                for slope, every in ((1.0, 1), (0.5, 2), (0.25, 4)):
                    rows[a == slope] = (steps > 0) & (steps % every == 0)
        elif case in ("late_spike", "spike_other_half"):
            gk = -4.0 * ((pos * 37) % T).to(f64) / T                # in [-4, 0], 0 at key 0
            gk[T - w + (5 if case == "late_spike" else w // 2 + 5)] = 20.0
            rows[:, nt - 1] = True
        else:
            a = torch.ones(T, dtype=f64)
            gk = -1.0 - 5.0 * ((pos * 37) % T).to(f64) / T
            gk[0] = 0.0
            gk[T // 2 + 3] = float(case.split("_")[1])
            if case == "threshold_8.5":
                rows[:, (T // 2 + 3) // w] = True
        q[..., 0] = a.view(1, T, 1)
        k[..., 0] = (gk / c).view(1, T, 1)
    return _pack(q, k, v, rows.expand(nsamp, heads, T, nt).clone(), f16, d, w, heads)


def _pack(q, k, v, expect, f16, d, w, heads):
    dt = torch.float16 if f16 else torch.bfloat16
    n, T = q.shape[:2]
    q, k, v = (x.reshape(n, T, heads * d).to(dt) for x in (q, k, v))
    return SimpleNamespace(q=q, k=k, v=v, expect=expect, d=d, w=w, heads=heads, scale=d ** -0.5, f16=f16)


def log2_logits(inp):
    n, T, _ = inp.q.shape
    qh, kh = (x.double().view(n, T, inp.heads, inp.d).transpose(1, 2) for x in (inp.q, inp.k))
    return (qh @ kh.transpose(2, 3)) * (inp.scale * LOG2E)


def score_magnitude(q, k, heads, scale):
    """scale * max_j (|Q| |K|^T)_ij per row, broadcast to the [n, T, heads * d] output layout."""
    n, T, Cc = q.shape
    d = Cc // heads
    qh = q.double().abs().view(n, T, heads, d).transpose(1, 2)
    kh = k.double().abs().view(k.shape[0], -1, heads, d).transpose(1, 2)
    m = (qh @ kh.transpose(2, 3)).amax(-1) * scale
    return m.transpose(1, 2).repeat_interleave(d, dim=-1)


def reference(q, k, v, heads, scale):
    """float64 O and A = softmax(scale Q K^T) |V| on the exact operand values (q [n, T, C], k / v [n, T, C])."""
    q, k, v = q.double(), k.double(), v.double()
    return O._mha_core(q, k, v, heads, scale), O._mha_core(q, k, v.abs(), heads, scale)


# ----------------------------------------------------------------------------------------------- CPU: the shadow of every case
@pytest.mark.parametrize("case", CASES)
def test_designed_inputs_reach_the_intended_rescales(case):
    for kernel in KERNELS:
        for f16 in (True, False):
            inp = make_case(case, kernel, 1024, f16)
            got, peak = shadow_rescales(log2_logits(inp), inp.w)
            assert torch.equal(got, inp.expect), (kernel, f16)
            assert bool(got.any()) == (case in RESCALING)
            if case == "threshold_7.5":
                assert 7.4 < float(peak.max()) < 7.6                # P reaches 2^7.5 under the stale maximum
            if case == "mixed_rows":                                # every warp has rows that rescale at a step and rows that do not
                per_warp = got.view(2, inp.heads, 1024 // 32, 32, -1)
                assert bool((per_warp.any(3) & ~per_warp.all(3)).any(-1).all())
            d = 2.0 ** -22 * score_magnitude(inp.q, inp.k, inp.heads, inp.scale)
            assert float(d.max()) < 2.0 ** -14, (kernel, float(d.max()))


def test_spikes_lie_in_the_intended_half_of_the_last_step():
    for kernel in KERNELS:
        w = tile_width(kernel, 1024)
        for case, half in (("late_spike", 0), ("spike_other_half", 1)):
            x = log2_logits(make_case(case, kernel, 1024, True))
            j = x.argmax(-1)
            assert bool((j // w == 1024 // w - 1).all()) and bool(((j % w) // (w // 2) == half).all())


@pytest.mark.parametrize("T", [128, 256, 384, 2048])
def test_sequence_length_inputs_reach_the_intended_rescales(T):
    for kernel in KERNELS:
        for case in ("ramp", "randn"):
            inp = make_case(case, kernel, T, False)
            got, _ = shadow_rescales(log2_logits(inp), inp.w)
            assert torch.equal(got, inp.expect) and bool(got.any()) == (case == "ramp")
            assert float(score_magnitude(inp.q, inp.k, inp.heads, inp.scale).max()) * 2.0 ** -22 < 2.0 ** -14


def test_shadow_rule_threshold_is_strict():
    x = torch.tensor([[0.0] * 4 + [8.0] * 4 + [16.5] * 4 + [17.0] * 4])
    got, peak = shadow_rescales(x, 4)
    assert got.tolist() == [[False, False, True, False]] and float(peak) == 8.0


# ----------------------------------------------------------------------------------------------- CPU: argument checks
def _hook(q, ldq, ks, ldk, vts, os_, olos, ldo, kv_div, nsamp, heads, T, d, scale, f16, nctx=None, stream=None):
    """dvd_test_attention_tc; pointers are tensors (their data_ptr), ints or None."""
    from dvd_b200 import _lib
    addr = lambda x: None if x is None else (x if isinstance(x, int) else x.data_ptr())
    arr = lambda xs: (C.c_void_p * len(xs))(*[addr(x) for x in xs])
    return _lib.lib().dvd_test_attention_tc(addr(q), ldq, arr(ks), ldk, arr(vts), arr(os_), None if olos is None else arr(olos), ldo,
                                            (C.c_int * len(kv_div))(*kv_div), len(ks) if nctx is None else nctx, nsamp, heads, T, d,
                                            scale, int(f16), stream)


def _last_error():
    from dvd_b200 import _lib
    return _lib.lib().dvd_last_error().decode()


_P = 1 << 24                  # a 16-byte aligned address: no call below gets as far as using it


def _bad_call(d=64, T=1024, nsamp=2, nctx=1, kv_div=None, ldo=None, o_off=0, lo_off=None, n_arr=None, heads=2):
    n_arr = n_arr or max(nctx, 1)
    kv = kv_div or [1] * n_arr
    ld = heads * d
    os_ = [_P + 0x100000 * i for i in range(n_arr)]
    os_[-1] += o_off
    los = None if lo_off is None else [_P + 0x800000 + 0x100000 * i for i in range(n_arr)]
    if los:
        los[-1] += lo_off
    return _hook(_P, ld, [_P] * n_arr, ld, [_P] * n_arr, os_, los, ld if ldo is None else ldo, kv, nsamp, heads, T, d, 0.125, True,
                 nctx=nctx)


ARG_CASES = {
    "nctx_0": (dict(nctx=0, n_arr=1), r"nctx must be 1\.\.4 \(got 0\)"),
    "nctx_5": (dict(nctx=5, n_arr=5), r"nctx must be 1\.\.4 \(got 5\)"),
    "d_128": (dict(d=128), r"bad shape d=128"),
    "d_128_4ctx": (dict(d=128, nctx=4), r"bad shape d=128"),
    "T_192_d64": (dict(T=192), r"bad shape d=64 T=192"),
    "T_192_d256": (dict(T=192, d=256), r"bad shape d=256 T=192"),
    "kv_div_tc": (dict(nsamp=3, kv_div=[2]), r"attention_tc: context 0: nsamp 3 is not a multiple of kv_div 2"),
    "kv_div_tc_4ctx": (dict(nsamp=3, nctx=4, kv_div=[1, 3, 2, 1]), r"context 2: nsamp 3 is not a multiple of kv_div 2"),
    "kv_div_pair": (dict(nsamp=3, kv_div=[2], d=256), r"attention_pair: nsamp 3 is not a multiple of kv_div 2"),
    "grid_tc": (dict(nsamp=65536), r"attention_tc: nsamp 65536 x nctx 1 exceeds 65535"),
    "grid_tc_4ctx": (dict(nsamp=16384, nctx=4), r"nsamp 16384 x nctx 4 exceeds 65535"),
    "grid_pair": (dict(nsamp=65536, d=256), r"attention_pair: nsamp 65536 outside 1\.\.65535"),
    "ldo_tc": (dict(ldo=132), r"attention_tc: ldo 132 is not a multiple of 8"),
    "ldo_pair": (dict(ldo=516, d=256), r"attention_pair: ldo 516 is not a multiple of 8"),
    "o_align_tc": (dict(o_off=8), r"attention_tc: context 0: o must be 16-byte aligned"),
    "o_align_tc_4ctx": (dict(o_off=8, nctx=4), r"context 3: o must be 16-byte aligned"),
    "o_align_pair": (dict(o_off=8, d=256), r"attention_pair: o must be 16-byte aligned"),
    "o_lo_align_tc": (dict(lo_off=2), r"attention_tc: context 0: o_lo must be 16-byte aligned"),
    "o_lo_align_tc_4ctx": (dict(lo_off=2, nctx=4), r"context 3: o_lo must be 16-byte aligned"),
    "o_lo_align_pair": (dict(lo_off=2, d=256), r"attention_pair: o_lo must be 16-byte aligned"),
}


@pytest.mark.parametrize("name", list(ARG_CASES))
def test_hook_rejects_bad_arguments_before_any_cuda_call(name, monkeypatch):
    """Every argument error comes back as DVD_E_BADARG with its own message; on a machine without a GPU any driver call (the
    tensor-map encode) would instead fail with DVD_E_NOTMA."""
    monkeypatch.delenv("DVD_ATTN_V1", raising=False)
    kw, msg = ARG_CASES[name]
    rc = _bad_call(**kw)
    err = _last_error()
    assert rc == DVD_E_BADARG and re.search(msg, err), (rc, err)


# ----------------------------------------------------------------------------------------------- GPU helpers
_RATIOS = {}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from dvd_b200 import _lib
    _lib.check(_lib.lib().dvd_check_device(), "dvd_check_device")
    yield torch.device("cuda:0")
    if _RATIOS:
        print("\nlargest error / bound:")
        for key in sorted(_RATIOS):
            print(f"  {key:24s} {_RATIOS[key]:.4f}")


def _select(kernel, monkeypatch):
    if KERNELS[kernel][1]:
        monkeypatch.setenv("DVD_ATTN_V1", "1")
    else:
        monkeypatch.delenv("DVD_ATTN_V1", raising=False)


class Arena:
    """`nreg` output regions [rows, ldo] inside one allocation, with slack before, between and after them, all prefilled with
    SENTINEL.  check() asserts that a launch wrote finite values to columns [0, cols) of the written regions and nothing else."""

    def __init__(self, dev, nreg, rows, ldo, cols, slack=4096):
        self.rows, self.ldo, self.cols = rows, ldo, cols
        self.off = [slack + r * (rows * ldo + slack) for r in range(nreg)]
        self.buf = torch.full((self.off[-1] + rows * ldo + slack,), SENTINEL, dtype=torch.int16, device=dev)

    def region(self, r):
        return self.buf[self.off[r]:self.off[r] + self.rows * self.ldo].view(self.rows, self.ldo)

    def ptr(self, r, row=0):
        return self.region(r)[row].data_ptr()

    def values(self, r):
        return self.region(r)[:, :self.cols].view(torch.bfloat16)

    def check(self, written):
        outside = torch.ones(self.buf.numel(), dtype=torch.bool, device=self.buf.device)
        for r in written:
            outside[self.off[r]:self.off[r] + self.rows * self.ldo].view(self.rows, self.ldo)[:, :self.cols] = False
            assert bool(torch.isfinite(self.values(r)).all()), f"region {r}: element not written or not finite"
        assert bool((self.buf[outside] == SENTINEL).all()), "a launch wrote outside its output regions"


def _check_bound(o, ref, A, mag, T, f16, with_lo, key):
    u_p = 2.0 ** -11 if f16 else 2.0 ** -8
    u_o = 2.0 ** -16 if with_lo else 2.0 ** -8
    bound = (2 * u_p + T * 2.0 ** -24 + 2.0 ** -22 * mag) * (A + ref.abs()) + u_o * ref.abs()
    _record(key, o, ref, bound)


def _record(key, o, ref, bound):
    assert bool(torch.isfinite(o).all())
    ratio = float(((o - ref).abs() / bound).max())
    _RATIOS[key] = max(_RATIOS.get(key, 0.0), ratio)
    assert ratio <= 1.0, f"{key}: error / bound = {ratio:.3f}"


def _run_designed(dev, inp, with_lo):
    """One launch of dvd_test_attention_tc on a designed case (ldo padded by 8 columns) -> O [n, T, C] float64."""
    from dvd_b200 import _lib
    n, T, Cc = inp.q.shape
    q, k, v = (x.to(dev) for x in (inp.q, inp.k, inp.v))
    vt = v.transpose(1, 2).contiguous()
    before = [x.clone() for x in (q, k, vt)]
    ldo = Cc + 8
    ar = Arena(dev, 2, n * T, ldo, Cc)
    rc = _hook(q, Cc, [k], Cc, [vt], [ar.ptr(0)], [ar.ptr(1)] if with_lo else None, ldo, [1], n, inp.heads, T, inp.d, inp.scale,
               inp.f16, stream=_lib.stream_ptr())
    _lib.check(rc, "dvd_test_attention_tc")
    torch.cuda.synchronize()
    ar.check([0, 1] if with_lo else [0])
    assert all(torch.equal(a, b) for a, b in zip(before, (q, k, vt)))
    o = ar.values(0).double()
    if with_lo:
        o = o + ar.values(1).double()
    return o.view(n, T, Cc), q, k, v


def _designed_vs_float64(dev, case, kernel, prec, T, monkeypatch):
    _select(kernel, monkeypatch)
    f16 = prec == "fp16"
    inp = make_case(case, kernel, T, f16)
    o, q, k, v = _run_designed(dev, inp, with_lo=f16)
    ref, A = reference(q, k, v, inp.heads, inp.scale)
    ran = kernel if inp.w == KERNELS[kernel][2] else "tc_d256"       # (the pair's fallback)
    _check_bound(o, ref, A, score_magnitude(q, k, inp.heads, inp.scale), T, f16, f16, f"{ran}/{prec}")


# ----------------------------------------------------------------------------------------------- GPU: the rescale branch
# fp16 operands with the hi + lo output pair (DVD_PREC_BF16X3), bf16 operands with the hi output alone (DVD_PREC_BF16)
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("case", CASES)
def test_rescale_cases_match_float64(dev, case, kernel, prec, monkeypatch):
    _designed_vs_float64(dev, case, kernel, prec, 1024, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("case", CASES)
def test_rescale_cases_fp32_path_match_float64(dev, case, kernel):
    """The same inputs (as fp32) through the fp32 attention of dvd_test_attention (precision 0)."""
    from dvd_b200 import _lib
    inp = make_case(case, kernel, 1024, True)
    n, T, Cc = inp.q.shape
    q, k, v = (x.float().to(dev) for x in (inp.q, inp.k, inp.v))
    o = torch.full_like(q, float("nan"))
    scratch = torch.empty(n * inp.heads * T * T * 4, dtype=torch.uint8, device=dev)
    _lib.check(_lib.lib().dvd_test_attention(_lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(o), n, inp.heads, T, inp.d, inp.scale, 0,
                                             _lib.ptr(scratch), scratch.numel(), _lib.stream_ptr()), "dvd_test_attention")
    torch.cuda.synchronize()
    ref, A = reference(q, k, v, inp.heads, inp.scale)
    mag = score_magnitude(q, k, inp.heads, inp.scale)
    bound = (2.0 ** -20 + 2 * T * 2.0 ** -24 + (inp.d + 2) * 2.0 ** -23 * mag) * (A + ref.abs())
    _record(f"fp32_path/d{inp.d}", o.double(), ref, bound)


# ----------------------------------------------------------------------------------------------- GPU: other sequence lengths
SEQ_PARAMS = [(kernel, T) for kernel in KERNELS for T in (128, 256, 384, 2048) if not (kernel == "pair_d256" and T == 128)]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("case", ["ramp", "randn"])
@pytest.mark.parametrize("kernel,T", SEQ_PARAMS)
def test_sequence_lengths_match_float64(dev, kernel, T, case, prec, monkeypatch):
    """T = 128 .. 2048 changes the number of key steps (the K / V ring phases and pv_done parities); pair_d256 at T = 384 is the
    default kernel choice for d = 256 falling back to k_attn_tc."""
    _designed_vs_float64(dev, case, kernel, prec, T, monkeypatch)


# ----------------------------------------------------------------------------------------------- GPU: the denoiser's launches
T_TOK = 1024


def _layout(kind, docs, n_hyp, dt, dev):
    """The operands in the denoiser's buffers.  Columns the attention must not read (V inside the packed buffers) hold NaN."""
    g = torch.Generator(device=dev).manual_seed(zlib.crc32(f"{kind}/{docs}/{n_hyp}".encode()))
    rnd = lambda *s: torch.randn(*s, generator=g, device=dev, dtype=torch.float32).to(dt)
    N = docs * n_hyp
    if kind == "cross":              # q [N*T, 384]; context i: K = columns 0..383 of [nkv*T, 768], V^T [nkv, 384, T]
        kv_div = (n_hyp, n_hyp, n_hyp, 1)
        kbufs = []
        for dv in kv_div:
            kv = rnd(N // dv * T_TOK, 768)
            kv[:, 384:] = float("nan")
            kbufs.append((kv, 0))
        return SimpleNamespace(nsamp=N, d=64, C=384, q=rnd(N * T_TOK, 384), kbufs=kbufs, ldk=768, kv_div=kv_div,
                               vts=[rnd(N // dv, 384, T_TOK) for dv in kv_div])
    if kind == "self":               # q | k | v in one [4N*T, 1152] buffer, K at +384; V^T [4N, 384, T]
        qkv = rnd(4 * N * T_TOK, 1152)
        qkv[:, 768:] = float("nan")
        return SimpleNamespace(nsamp=4 * N, d=64, C=384, q=qkv, kbufs=[(qkv, 384)], ldk=1152, kv_div=(1,), vts=[rnd(4 * N, 384, T_TOK)])
    qkv = rnd(N * T_TOK, 4608)       # decoder: [N*T, 4608], K at +1536; V^T [N, 1536, T]
    qkv[:, 3072:] = float("nan")
    return SimpleNamespace(nsamp=N, d=256, C=1536, q=qkv, kbufs=[(qkv, 1536)], ldk=4608, kv_div=(1,), vts=[rnd(N, 1536, T_TOK)])


def _checked_samples(nsamp, n_hyp):
    if nsamp <= 8:
        return list(range(nsamp))
    return sorted({0, 1, n_hyp - 1, nsamp // 2, nsamp // 2 + 1, nsamp - n_hyp, nsamp - 1})


def _layout_test(dev, kind, docs, n_hyp, prec, monkeypatch):
    from dvd_b200 import _lib
    monkeypatch.delenv("DVD_ATTN_V1", raising=False)
    f16 = prec == "fp16"
    L = _layout(kind, docs, n_hyp, torch.float16 if f16 else torch.bfloat16, dev)
    n, nctx, Cc, ldq = L.nsamp, len(L.kv_div), L.C, L.q.shape[1]
    heads, scale = Cc // L.d, L.d ** -0.5
    rows = n * T_TOK
    st = _lib.stream_ptr()

    def launch(arena, samples, nb, kv_div):
        s0 = samples[0]
        ks = [kb[(s0 // dv) * T_TOK, off].data_ptr() for (kb, off), dv in zip(L.kbufs, L.kv_div)]
        vts = [vt[s0 // dv].data_ptr() for vt, dv in zip(L.vts, L.kv_div)]
        los = [arena.ptr(nctx + i, s0 * T_TOK) for i in range(nctx)] if f16 else None
        _lib.check(_hook(L.q[s0 * T_TOK].data_ptr(), ldq, ks, L.ldk, vts, [arena.ptr(i, s0 * T_TOK) for i in range(nctx)], los, Cc,
                         kv_div, nb, heads, T_TOK, L.d, scale, f16, stream=st), "dvd_test_attention_tc")

    batch = Arena(dev, 2 * nctx, rows, Cc, Cc)
    launch(batch, [0], n, L.kv_div)
    single = Arena(dev, 2 * nctx, rows, Cc, Cc)
    for s in range(n):                                              # the same operands, one sample per launch (kv_div 1)
        launch(single, [s], 1, [1] * nctx)
    torch.cuda.synchronize()
    written = list(range(2 * nctx)) if f16 else list(range(nctx))
    batch.check(written)
    single.check(written)
    assert torch.equal(batch.buf, single.buf), "a batched launch differs from one-sample launches of the same operands"
    for s in _checked_samples(n, n_hyp):
        for i in range(nctx):
            kb, off = L.kbufs[i]
            kv = s // L.kv_div[i]
            q = L.q[s * T_TOK:(s + 1) * T_TOK, :Cc].unsqueeze(0)
            k = kb[kv * T_TOK:(kv + 1) * T_TOK, off:off + Cc].unsqueeze(0)
            v = L.vts[i][kv].t().unsqueeze(0)
            ref, A = reference(q, k, v, heads, scale)
            o = batch.values(i)[s * T_TOK:(s + 1) * T_TOK].double()
            if f16:
                o = o + batch.values(nctx + i)[s * T_TOK:(s + 1) * T_TOK].double()
            key = f"{'pair_d256' if L.d == 256 else 'tc_d64'}/{prec}"
            _check_bound(o.unsqueeze(0), ref, A, score_magnitude(q, k, heads, scale), T_TOK, f16, f16, key)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("docs,n_hyp", [(1, 2), (3, 3), (16, 2)])
def test_dit_cross_attention_four_contexts(dev, docs, n_hyp, prec, monkeypatch):
    """One four-context launch over shared queries, K / V of the three static contexts shared by each document's hypotheses."""
    _layout_test(dev, "cross", docs, n_hyp, prec, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("docs,n_hyp", [(1, 2), (3, 3), (16, 2), (64, 2)])
def test_dit_self_attention_packed_qkv(dev, docs, n_hyp, prec, monkeypatch):
    """4 * docs * n_hyp samples (up to 512: grid z = 512) with Q and K inside one packed q | k | v buffer."""
    _layout_test(dev, "self", docs, n_hyp, prec, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("docs,n_hyp", [(1, 2), (3, 3), (16, 2)])
def test_decoder_attention_packed_qkv(dev, docs, n_hyp, prec, monkeypatch):
    """Head dim 256 on the CTA-pair kernel, Q and K inside the decoder's [N*T, 4608] q | k | v buffer."""
    _layout_test(dev, "decoder", docs, n_hyp, prec, monkeypatch)
