"""CPU ORACLE for the GPU JPEG decoder (TEST INFRASTRUCTURE, NOT PRODUCT CODE).

The reference loader reads a photo as ``cv2.imread(path)[..., ::-1]`` (datasets/doc_dataset/doc_benchmark.py:68-71 in the
reference): libjpeg-turbo's default decode, then the EXIF orientation OpenCV applies.  This restates that decode of baseline /
extended sequential 8-bit Huffman files with one interleaved scan in numpy plus a plain Python Huffman loop, so that the GPU
kernels (dvd_b200/csrc/jpeg.cu) can be checked without the library:

  * entropy decode (jdhuff.c): DC prediction per component, reset at every restart marker; AC run/size symbols in zigzag order
  * dequantize + jpeg_idct_islow (jidctint.c, CONST_BITS 13, PASS1_BITS 2), output through the post-IDCT range-limit table of
    jdmaster.c, indexed with & 1023: clamp(sign_extend_10(v) + 128, 0, 255)
  * "fancy" upsampling (jdsample.c) of chroma with h = 2 (4:2:2: v = 1, 4:2:0: v = 2); the edges replicate the component's last
    real sample (index ceil(W * h / hmax) - 1), and rows are read across MCU-row boundaries.  A component at most 2 samples wide
    is upsampled by replication instead (jinit_upsampler picks fancy only for downsampled_width > 2)
  * ycc_rgb_convert (jdcolor.c) with its 16-bit fixed-point tables; grayscale is replicated to three channels
  * the EXIF orientation (APP1, IFD0 tag 0x0112, either byte order) as OpenCV's transpose / flip
"""
from __future__ import annotations

import numpy as np

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
                   28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61,
                   54, 47, 55, 62, 63])
# libjpeg's jpeg_natural_order has 16 extra entries so that a corrupt run past 63 lands on 63
NATURAL = np.concatenate([ZIGZAG, np.full(16, 63)])


def exif_orientation(buf: bytes) -> int:
    """orientation 1..8 from the first APP1 Exif segment (1 when absent or malformed)"""
    i = 2
    while i + 4 <= len(buf) and buf[i] == 0xFF:
        m, ln = buf[i + 1], int.from_bytes(buf[i + 2:i + 4], "big")
        if m == 0xDA:
            break
        seg = buf[i + 4:i + 2 + ln]
        if m == 0xE1 and seg[:6] == b"Exif\0\0":
            t = seg[6:]
            if len(t) < 8 or t[:2] not in (b"II", b"MM"):
                return 1
            bo = "little" if t[:2] == b"II" else "big"
            ifd = int.from_bytes(t[4:8], bo)
            if ifd + 2 > len(t):
                return 1
            for e in range(int.from_bytes(t[ifd:ifd + 2], bo)):
                p = ifd + 2 + 12 * e
                if p + 12 > len(t):
                    return 1
                if int.from_bytes(t[p:p + 2], bo) == 0x0112:
                    v = int.from_bytes(t[p + 8:p + 10], bo)
                    return v if 1 <= v <= 8 else 1
            return 1
        i += 2 + ln
    return 1


def _parse(buf: bytes):
    q, dc, ac, comps, ri = {}, {}, {}, None, 0
    i = 2
    while True:
        while buf[i] == 0xFF and buf[i + 1] == 0xFF:
            i += 1
        m, ln = buf[i + 1], int.from_bytes(buf[i + 2:i + 4], "big")
        seg = buf[i + 4:i + 2 + ln]
        if m == 0xDB:
            p = 0
            while p < len(seg):
                pq, tq = seg[p] >> 4, seg[p] & 15
                n = 128 if pq else 64
                vals = np.frombuffer(seg[p + 1:p + 1 + n], ">u2" if pq else "u1").astype(np.int64)
                nat = np.zeros(64, np.int64)
                nat[ZIGZAG] = vals
                q[tq] = nat
                p += 1 + n
        elif m == 0xC4:
            p = 0
            while p < len(seg):
                tc, th = seg[p] >> 4, seg[p] & 15
                counts = list(seg[p + 1:p + 17])
                vals = list(seg[p + 17:p + 17 + sum(counts)])
                (ac if tc else dc)[th] = _lut(counts, vals)
                p += 17 + sum(counts)
        elif m in (0xC0, 0xC1):
            H, W = int.from_bytes(seg[1:3], "big"), int.from_bytes(seg[3:5], "big")
            comps = [dict(id=seg[6 + 3 * c], h=seg[7 + 3 * c] >> 4, v=seg[7 + 3 * c] & 15, tq=seg[8 + 3 * c]) for c in range(seg[5])]
        elif m == 0xDD:
            ri = int.from_bytes(seg[0:2], "big")
        elif m == 0xDA:
            for c in range(seg[0]):
                cid, t = seg[1 + 2 * c], seg[2 + 2 * c]
                comp = next(x for x in comps if x["id"] == cid)
                comp["td"], comp["ta"] = t >> 4, t & 15
            return H, W, comps, q, dc, ac, ri, i + 2 + ln
        i += 2 + ln


class _Bits:
    """the entropy-coded segments of a scan: bytes with 0xFF00 destuffed, split at RSTn markers"""

    def __init__(self, buf: bytes, start: int):
        segs, cur, i = [], bytearray(), start
        while True:
            b = buf[i]
            if b != 0xFF:
                cur.append(b)
                i += 1
                continue
            while buf[i + 1] == 0xFF:
                i += 1
            nb = buf[i + 1]
            if nb == 0:
                cur.append(0xFF)
                i += 2
            elif 0xD0 <= nb <= 0xD7:
                segs.append(bytes(cur))
                cur = bytearray()
                i += 2
            else:
                segs.append(bytes(cur))
                break
        self.segs = segs

    def start(self, k):
        self.b = (self.segs[k] if k < len(self.segs) else b"") + bytes(8)     # past the data libjpeg feeds zeros
        self.pos = 0

    def peek16(self):
        p, b = self.pos >> 3, self.b
        if p + 3 > len(b):
            return 0
        return ((b[p] << 16 | b[p + 1] << 8 | b[p + 2]) >> (8 - (self.pos & 7))) & 0xFFFF

    def get(self, n):
        v = self.peek16() >> (16 - n) if n else 0
        self.pos += n
        return v

    def sym(self, lut):
        ln, s = lut[self.peek16()]
        self.pos += ln
        return s


def _lut(counts, vals):
    """(length, symbol) for every 16-bit window; a bad code decodes as symbol 0 and consumes 16 bits (jdhuff.c JWRN_HUFF_BAD_CODE)"""
    lut = [(16, 0)] * 65536
    code, k = 0, 0
    for l in range(1, 17):
        for _ in range(counts[l - 1]):
            lo = code << (16 - l)
            lut[lo:lo + (1 << (16 - l))] = [(l, vals[k])] * (1 << (16 - l))
            code += 1
            k += 1
        code <<= 1
    return lut


def _extend(r, s):
    return r - (1 << s) + 1 if s and r < (1 << (s - 1)) else r


def decode_coefficients(buf: bytes):
    """header fields and the quantized coefficients [component] -> int64 [blocks_y, blocks_x, 64] (natural order)"""
    H, W, comps, q, dc, ac, ri, scan = _parse(buf)
    hmax, vmax = max(c["h"] for c in comps), max(c["v"] for c in comps)
    if len(comps) == 1:                            # a non-interleaved scan: one block per MCU, blocks of the component only
        comps[0]["h"] = comps[0]["v"] = hmax = vmax = 1
        mcux, mcuy = -(-W // 8), -(-H // 8)
    else:
        mcux, mcuy = -(-W // (8 * hmax)), -(-H // (8 * vmax))
    coef = [np.zeros((mcuy * c["v"], mcux * c["h"], 64), np.int64) for c in comps]
    bits = _Bits(buf, scan)
    total = mcux * mcuy
    per = ri if ri else total
    for seg in range(-(-total // per)):
        bits.start(seg)
        pred = [0] * len(comps)
        for m in range(seg * per, min(total, (seg + 1) * per)):
            my, mx = divmod(m, mcux)
            for ci, c in enumerate(comps):
                for by in range(c["v"]):
                    for bx in range(c["h"]):
                        blk = coef[ci][my * c["v"] + by, mx * c["h"] + bx]
                        s = bits.sym(dc[c["td"]])
                        pred[ci] += _extend(bits.get(s), s)
                        blk[0] = np.int16(pred[ci])           # JCOEF is 16-bit; the predictor itself is an int
                        k = 1
                        while k < 64:
                            rs = bits.sym(ac[c["ta"]])
                            r, s = rs >> 4, rs & 15
                            if s:
                                k += r
                                blk[NATURAL[k]] = _extend(bits.get(s), s)
                            elif r != 15:
                                break
                            else:
                                k += 15
                            k += 1
    return H, W, comps, hmax, vmax, q, coef


_C = {"0_298631336": 2446, "0_390180644": 3196, "0_541196100": 4433, "0_765366865": 6270, "0_899976223": 7373,
      "1_175875602": 9633, "1_501321110": 12299, "1_847759065": 15137, "1_961570560": 16069, "2_053119869": 16819,
      "2_562915447": 20995, "3_072711026": 25172}


def _idct_1d(x, shift):
    """one pass of jpeg_idct_islow over axis -2 of int64 x [..., 8, 8]; returns DESCALE(., shift)"""
    F = _C
    r = lambda k: x[..., k, :]
    z2, z3 = r(2), r(6)
    z1 = (z2 + z3) * F["0_541196100"]
    tmp2 = z1 + z3 * -F["1_847759065"]
    tmp3 = z1 + z2 * F["0_765366865"]
    tmp0 = (r(0) + r(4)) << 13
    tmp1 = (r(0) - r(4)) << 13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    tmp0, tmp1, tmp2, tmp3 = r(7), r(5), r(3), r(1)
    z1, z2, z3, z4 = tmp0 + tmp3, tmp1 + tmp2, tmp0 + tmp2, tmp1 + tmp3
    z5 = (z3 + z4) * F["1_175875602"]
    tmp0, tmp1, tmp2, tmp3 = tmp0 * F["0_298631336"], tmp1 * F["2_053119869"], tmp2 * F["3_072711026"], tmp3 * F["1_501321110"]
    z1, z2 = z1 * -F["0_899976223"], z2 * -F["2_562915447"]
    z3, z4 = z3 * -F["1_961570560"] + z5, z4 * -F["0_390180644"] + z5
    tmp0, tmp1, tmp2, tmp3 = tmp0 + z1 + z3, tmp1 + z2 + z4, tmp2 + z2 + z3, tmp3 + z1 + z4
    d = lambda v: (v + (1 << (shift - 1))) >> shift
    out = [t10 + tmp3, t11 + tmp2, t12 + tmp1, t13 + tmp0, t13 - tmp0, t12 - tmp1, t11 - tmp2, t10 - tmp3]
    return np.stack([d(v) for v in out], axis=-2)


def idct_islow(coef, qt):
    """uint8 samples [..., 8, 8] of int64 coefficient blocks [..., 64] (natural order) and their table [64]"""
    x = (coef * qt).reshape(coef.shape[:-1] + (8, 8))
    ws = _idct_1d(x, 13 - 2)                                         # columns
    out = _idct_1d(np.swapaxes(ws, -1, -2), 13 + 2 + 3)              # rows (transposed back below)
    v = np.swapaxes(out, -1, -2) & 1023
    return np.clip(np.where(v < 512, v, v - 1024) + 128, 0, 255).astype(np.int64)


def _planes(H, W, comps, hmax, vmax, q, coef):
    planes = []
    for c, k in zip(comps, coef):
        s = idct_islow(k, q[c["tq"]])                                # [by, bx, 8, 8]
        p = s.transpose(0, 2, 1, 3).reshape(s.shape[0] * 8, s.shape[1] * 8)
        planes.append(p[:-(-H * c["v"] // vmax), :-(-W * c["h"] // hmax)])      # the component's real samples
    return planes


def _up_h2(a, rounding):
    """fancy horizontal doubling of the last axis: (3 near + far + rounding[parity]) >> shift, with replicated edges"""
    left = np.concatenate([a[..., :1], a[..., :-1]], axis=-1)
    right = np.concatenate([a[..., 1:], a[..., -1:]], axis=-1)
    out = np.empty(a.shape[:-1] + (2 * a.shape[-1],), np.int64)
    out[..., 0::2] = 3 * a + left + rounding[0]
    out[..., 1::2] = 3 * a + right + rounding[1]
    return out


def _upsample(p, h, v, H, W):
    if h == 1 and v == 1:
        return p
    if p.shape[1] <= 2:                                               # jdsample.c: fancy only when downsampled_width > 2
        return np.repeat(np.repeat(p, v, axis=0), 2, axis=1)[:H, :W]
    if v == 1:                                                        # h2v1
        return (_up_h2(p, (1, 2)) >> 2)[:H, :W]
    up = np.concatenate([p[:1], p[:-1]], axis=0)                      # h2v2: column sums 3 near + far, rows replicated
    dn = np.concatenate([p[1:], p[-1:]], axis=0)
    cs = np.empty((2 * p.shape[0], p.shape[1]), np.int64)
    cs[0::2] = 3 * p + up
    cs[1::2] = 3 * p + dn
    return (_up_h2(cs, (8, 7)) >> 4)[:H, :W]


def _ycc_rgb(y, cb, cr):
    fix = lambda x: int(x * 65536 + 0.5)
    x = np.arange(256, dtype=np.int64) - 128
    cr_r = (fix(1.40200) * x + 32768) >> 16
    cb_b = (fix(1.77200) * x + 32768) >> 16
    cr_g = -fix(0.71414) * x
    cb_g = -fix(0.34414) * x + 32768
    r = y + cr_r[cr]
    g = y + ((cb_g[cb] + cr_g[cr]) >> 16)
    b = y + cb_b[cb]
    return np.clip(np.stack([r, g, b], axis=-1), 0, 255)


def orient(img: np.ndarray, o: int) -> np.ndarray:
    """OpenCV's EXIF transform: 2 flip x, 3 flip both, 4 flip y, 5 transpose, 6 transpose + flip x, 7 transpose + flip both,
    8 transpose + flip y"""
    if o >= 5:
        img = img.transpose(1, 0, 2)
    flip = {2: (1,), 3: (0, 1), 4: (0,), 6: (1,), 7: (0, 1), 8: (0,)}.get(o, ())
    return np.flip(img, flip) if flip else img


def decode(buf: bytes) -> np.ndarray:
    """uint8 HWC RGB, equal to cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR)[..., ::-1]"""
    buf = bytes(buf)
    H, W, comps, hmax, vmax, q, coef = decode_coefficients(buf)
    planes = _planes(H, W, comps, hmax, vmax, q, coef)
    if len(comps) == 1:
        rgb = np.repeat(planes[0][:, :, None], 3, axis=2)
    else:
        y = planes[0][:H, :W]
        cb, cr = (_upsample(p, hmax // c["h"], vmax // c["v"], H, W) for p, c in zip(planes[1:], comps[1:]))
        rgb = _ycc_rgb(y, cb, cr)
    return np.ascontiguousarray(orient(rgb.astype(np.uint8), exif_orientation(buf)))
