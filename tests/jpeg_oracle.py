"""CPU reference of the library's JPEG encoder (test infrastructure): libjpeg's default baseline at quality q — JFIF,
4:2:0, the standard Huffman tables of ITU-T T.81 Annex K, no restart markers — restated step by step in integer numpy.

oracle_jpeg(rgb, w, h, quality) returns the bytes PIL.Image.save(format="JPEG", quality=q) writes for the same frame;
tests/test_jpeg.py checks that on the CPU, and the device encoder (rt_jpeg_encode) against both.
"""
from __future__ import annotations

import numpy as np

ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
    62, 63], dtype=np.int64)  # zigzag index -> natural (row-major) index

# Annex K.1 base quantisation tables, natural order
BASE_LUMA = [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22,
             29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103,
             121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99]
BASE_CHROMA = [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66,
               99, 99, 99, 99, 99, 99] + [99] * 32

# Annex K.3 Huffman tables: (code counts per length 1..16, symbols in code order)
DC_LUMA = ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12)))
DC_CHROMA = ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12)))
AC_LUMA = ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125], bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f0243362728209"
    "0a161718191a25262728292a3435363738393a434445464748494a535455565758595a636465"
    "666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9"
    "aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9ea"
    "f1f2f3f4f5f6f7f8f9fa"))
AC_CHROMA = ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119], bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a16"
    "2434e125f11718191a262728292a35363738393a434445464748494a535455565758595a6364"
    "65666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7"
    "a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9"
    "eaf2f3f4f5f6f7f8f9fa"))


def quant_tables(quality: int):
    """jpeg_quality_scaling + jpeg_add_quant_table (force_baseline): natural order, 1..255."""
    q = min(max(int(quality), 1), 100)
    scale = 5000 // q if q < 50 else 200 - 2 * q
    out = []
    for base in (BASE_LUMA, BASE_CHROMA):
        out.append(np.array([min(max((b * scale + 50) // 100, 1), 255) for b in base], dtype=np.int64))
    return out


def huff_codes(table):
    """Canonical codes (Annex C): symbol -> (code, length)."""
    bits, vals = table
    codes, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return codes


def header(w: int, h: int, quality: int) -> bytes:
    """SOI, APP0 (JFIF 1.01), DQT x2, SOF0 (4:2:0), DHT x4, SOS: 623 bytes."""
    def seg(marker, body):
        return bytes([0xFF, marker]) + (len(body) + 2).to_bytes(2, "big") + body

    qt = quant_tables(quality)
    out = b"\xff\xd8" + seg(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for i in (0, 1):
        out += seg(0xDB, bytes([i]) + bytes(int(v) for v in qt[i][ZIGZAG]))
    out += seg(0xC0, bytes([8]) + h.to_bytes(2, "big") + w.to_bytes(2, "big") + bytes([3, 1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
    for tc, t in ((0x00, DC_LUMA), (0x10, AC_LUMA), (0x01, DC_CHROMA), (0x11, AC_CHROMA)):
        out += seg(0xC4, bytes([tc]) + bytes(t[0]) + bytes(t[1]))
    out += seg(0xDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0]))
    return out


def _fix(x):
    return int(x * 65536 + 0.5)


def ycc(rgb):
    """rgb_ycc_convert (jccolor.c): 16-bit fixed point, int64 planes."""
    r, g, b = (rgb[..., i].astype(np.int64) for i in range(3))
    half = 1 << 15
    y = (_fix(0.29900) * r + _fix(0.58700) * g + _fix(0.11400) * b + half) >> 16
    cb = (-_fix(0.16874) * r - _fix(0.33126) * g + _fix(0.5) * b + (128 << 16) + half - 1) >> 16
    cr = (_fix(0.5) * r - _fix(0.41869) * g - _fix(0.08131) * b + (128 << 16) + half - 1) >> 16
    return y, cb, cr


def fdct_islow(blocks):
    """jpeg_fdct_islow (jfdctint.c) over (..., 8, 8) int64 samples already centred on 0; output scaled by 8."""
    CB, P1 = 13, 2
    F = dict(c0298=2446, c0390=3196, c0541=4433, c0765=6270, c0899=7373, c1175=9633, c1501=12299, c1847=15137,
             c1961=16069, c2053=16819, c2562=20995, c3072=25172)

    def descale(x, n):
        return (x + (1 << (n - 1))) >> n

    def pass_(d, first):
        d = [d[..., i] for i in range(8)]
        t0, t7 = d[0] + d[7], d[0] - d[7]
        t1, t6 = d[1] + d[6], d[1] - d[6]
        t2, t5 = d[2] + d[5], d[2] - d[5]
        t3, t4 = d[3] + d[4], d[3] - d[4]
        t10, t13 = t0 + t3, t0 - t3
        t11, t12 = t1 + t2, t1 - t2
        o = [None] * 8
        n = CB - P1 if first else CB + P1
        if first:
            o[0], o[4] = (t10 + t11) << P1, (t10 - t11) << P1
        else:
            o[0], o[4] = descale(t10 + t11, P1), descale(t10 - t11, P1)
        z1 = (t12 + t13) * F["c0541"]
        o[2] = descale(z1 + t13 * F["c0765"], n)
        o[6] = descale(z1 - t12 * F["c1847"], n)
        z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
        z5 = (z3 + z4) * F["c1175"]
        t4, t5, t6, t7 = t4 * F["c0298"], t5 * F["c2053"], t6 * F["c3072"], t7 * F["c1501"]
        z1, z2 = -z1 * F["c0899"], -z2 * F["c2562"]
        z3, z4 = -z3 * F["c1961"] + z5, -z4 * F["c0390"] + z5
        o[7] = descale(t4 + z1 + z3, n)
        o[5] = descale(t5 + z2 + z4, n)
        o[3] = descale(t6 + z2 + z3, n)
        o[1] = descale(t7 + z1 + z4, n)
        return np.stack(o, axis=-1)

    rows = pass_(blocks, True)                                  # over each row
    return np.swapaxes(pass_(np.swapaxes(rows, -1, -2), False), -1, -2)  # over each column


def quantise(coef, qt):
    """Divide by 8 * quantval, magnitude rounded half up (jcdctmgr.c quantize)."""
    d = qt.reshape(8, 8) * 8
    mag = np.abs(coef)
    q = np.where(mag < d // 2, 0, (mag + d // 2) // d)
    return np.where(coef < 0, -q, q)


def _blocks(plane, by, bx):
    """(by*8, bx*8) plane -> (by, bx, 8, 8) blocks."""
    return plane.reshape(by, 8, bx, 8).swapaxes(1, 2)


def mcu_blocks(rgb, w, h, quality):
    """Quantised coefficients in zigzag order, (mcu_rows, mcu_cols, 6, 64): Y00 Y01 Y10 Y11 Cb Cr per MCU."""
    mx, my = -(-w // 16), -(-h // 16)
    bw, bh = -(-w // 8), -(-h // 8)  # luma blocks that hold image data; the others of a partial MCU are dummies
    qt = quant_tables(quality)
    # luma: columns past w repeat column w-1, rows past h repeat row h-1
    ys = np.minimum(np.arange(16 * my), h - 1)
    xs = np.minimum(np.arange(16 * mx), w - 1)
    y, _, _ = ycc(rgb[ys][:, xs])
    # chroma: rows padded to an even count (row h-1 repeated), columns to 16 * mx; 2x2 sums with the bias 1, 2, 1, 2 ...
    hc = -(-h // 2)
    _, cb, cr = ycc(rgb[np.minimum(np.arange(2 * hc), h - 1)][:, xs])
    bias = np.tile([1, 2], 4 * mx)
    chroma = []
    for c in (cb, cr):
        s = c[0::2, 0::2] + c[0::2, 1::2] + c[1::2, 0::2] + c[1::2, 1::2]
        s = (s + bias) >> 2
        # rows past ceil(h/2) repeat the last downsampled row
        chroma.append(s[np.minimum(np.arange(8 * my), hc - 1)])

    def dct_quant(plane, by, bx, table):
        c = quantise(fdct_islow(_blocks(plane - 128, by, bx)), table)
        return c.reshape(by, bx, 64)[..., ZIGZAG]

    Y = dct_quant(y, 2 * my, 2 * mx, qt[0])
    Cb = dct_quant(chroma[0], my, mx, qt[1])
    Cr = dct_quant(chroma[1], my, mx, qt[1])
    # dummy luma blocks: all zero, DC copied from the block before in MCU order (jccoefct.c compress_data)
    if bw % 2:
        Y[:, bw] = 0
        Y[:, bw, 0] = Y[:, bw - 1, 0]
    if bh % 2:
        Y[bh] = 0
        Y[bh, 0::2, 0] = Y[bh - 1, 1::2, 0]
        Y[bh, 1::2, 0] = Y[bh - 1, 1::2, 0]
    Y = Y.reshape(my, 2, mx, 2, 64).transpose(0, 2, 1, 3, 4).reshape(my, mx, 4, 64)
    return np.concatenate([Y, Cb[:, :, None], Cr[:, :, None]], axis=2)


def _bit_size(v):
    """Bits of |v| (0 for 0)."""
    a = np.abs(v)
    n = np.zeros(a.shape, dtype=np.int64)
    while True:
        m = a >> n > 0
        if not m.any():
            return n
        n += m


def entropy_code(blocks) -> bytes:
    """The scan of (mcus, 6, 64) zigzag blocks: Huffman coded, padded with 1-bits, 0xFF followed by 0x00."""
    nb = blocks.shape[0] * 6
    z = blocks.reshape(nb, 64).astype(np.int64)
    comp = np.tile([0, 0, 0, 0, 1, 2], blocks.shape[0])
    # DC predictor per component across the whole scan, starting at 0
    diff = np.empty(nb, dtype=np.int64)
    for c in range(3):
        idx = np.nonzero(comp == c)[0]
        dc = z[idx, 0]
        diff[idx] = dc - np.concatenate([[0], dc[:-1]])
    chroma = comp > 0
    tables = [(huff_codes(DC_LUMA), huff_codes(AC_LUMA)), (huff_codes(DC_CHROMA), huff_codes(AC_CHROMA))]

    def lookup(symbols, is_chroma, ac):
        code = np.empty(symbols.shape, dtype=np.int64)
        length = np.empty(symbols.shape, dtype=np.int64)
        for t in (0, 1):
            m = is_chroma == bool(t)
            tab = tables[t][1 if ac else 0]
            code[m] = [tab[int(s)][0] for s in symbols[m]]
            length[m] = [tab[int(s)][1] for s in symbols[m]]
        return code, length

    def magnitude_bits(v, n):  # a negative value's bits are v - 1 masked to its size
        return np.where(v < 0, v - 1, v) & ((np.int64(1) << n) - 1)

    # one item (value, length, block, position) per DC, per nonzero AC (with its leading ZRLs folded in) and per EOB
    n = _bit_size(diff)
    code, length = lookup(n, chroma, False)
    items = [(code << n | magnitude_bits(diff, n), length + n, np.arange(nb), np.zeros(nb, dtype=np.int64))]
    b, k = np.nonzero(z[:, 1:])
    k = k + 1
    v = z[b, k]
    first = np.ones(len(b), dtype=bool)
    first[1:] = b[1:] != b[:-1]
    prev = np.where(first, 0, np.concatenate([[0], k[:-1]]))
    run = k - prev - 1
    n = _bit_size(v)
    code, length = lookup((run & 15) << 4 | n, chroma[b], True)
    zrl_code, zrl_len = lookup(np.full(len(b), 0xF0), chroma[b], True)
    val, ln = np.zeros(len(b), dtype=np.int64), np.zeros(len(b), dtype=np.int64)
    for _ in range(3):  # at most 3 runs of 16 zeros before a nonzero coefficient
        m = run >= 16 * (_ + 1)
        val = np.where(m, val << zrl_len | zrl_code, val)
        ln = np.where(m, ln + zrl_len, ln)
    val = ((val << length | code) << n) | magnitude_bits(v, n)
    items.append((val, ln + length + n, b, k))
    last = np.zeros(nb, dtype=np.int64)
    np.maximum.at(last, b, k)
    eob = np.nonzero(last < 63)[0]
    code, length = lookup(np.zeros(len(eob), dtype=np.int64), chroma[eob], True)
    items.append((code, length, eob, np.full(len(eob), 64)))

    val, ln, blk, pos = (np.concatenate(x) for x in zip(*items))
    order = np.lexsort((pos, blk))
    val, ln = val[order].astype(np.uint64), ln[order]
    # pack MSB first into 64-bit words; an item (<= 59 bits) spans at most two words
    off = np.concatenate([[0], np.cumsum(ln)[:-1]])
    total = int(ln.sum())
    words = np.zeros(total // 64 + 2, dtype=np.uint64)
    wi, s = off // 64, off % 64
    end = s + ln
    fits = end <= 64
    sh = np.where(fits, 64 - end, 0).astype(np.uint64)
    np.bitwise_or.at(words, wi[fits], val[fits] << sh[fits])
    sp = ~fits
    hi = (end[sp] - 64).astype(np.uint64)
    np.bitwise_or.at(words, wi[sp], val[sp] >> hi)
    np.bitwise_or.at(words, wi[sp] + 1, val[sp] << (np.uint64(64) - hi))
    data = bytearray(words.byteswap().tobytes()[: (total + 7) // 8])
    if total % 8:
        data[-1] |= (1 << (8 - total % 8)) - 1
    return bytes(data).replace(b"\xff", b"\xff\x00")


def oracle_jpeg(rgb, w: int, h: int, quality: int = 90) -> bytes:
    """Baseline JPEG of an RGB8 frame (h, w, 3), byte-identical to libjpeg's defaults at this quality."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8).reshape(h, w, 3)
    blocks = mcu_blocks(rgb, w, h, quality)
    return header(w, h, quality) + entropy_code(blocks.reshape(-1, 6, 64)) + b"\xff\xd9"
