"""Reference JPEG decode (numpy restatement of libjpeg 6.2 as Pillow runs it) from the ``EncodedImages`` representation.

Sequential Huffman decode bit by bit with the canonical maxcode / valoffset form (no lookahead table), DC prediction
restarting at every interval, dequantisation and the integer "islow" IDCT (CONST_BITS 13, PASS1_BITS 2, libjpeg's
range-limit table), fancy (triangle) upsampling for 2x1 / 2x2 chroma wider than 2 samples (else replication), and the
fixed-point YCbCr -> RGB of jdcolor.c.  Test infrastructure only: nothing under the package imports it.
"""
import numpy as np

NATURAL = np.array(list(np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                                  13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59,
                                  52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])) + [63] * 16)


def _huff(tables, off):
    rec = tables[off:off + 1024]
    return rec[512:584].view(np.int32), rec[584:656].view(np.int32), rec[656:912]


def _decode_symbol(bits, p, table):
    maxcode, valoff, huffval = table
    code, length = 0, 0
    while True:
        code = (code << 1) | (int(bits[p]) if p < len(bits) else 0)
        p += 1
        length += 1
        if length > 16:
            return 0, p
        if code <= maxcode[length]:
            return int(huffval[(code + int(valoff[length])) & 255]), p


def _receive(bits, p, s):
    v = 0
    for _ in range(s):
        v = (v << 1) | (int(bits[p]) if p < len(bits) else 0)
        p += 1
    if s and v < (1 << (s - 1)):
        v += (-1 << s) + 1
    return v, p


def entropy_decode(enc, i):
    """Coefficients of image i: per component int64 [blocks_y, blocks_x, 64] (natural order, DC absolute), padded to whole
    MCUs, and the geometry (ncomp, hmax, vmax, mcus_x, mcus_y)."""
    d = [int(v) for v in enc.desc[i]]
    data, tables = enc.data.numpy(), enc.tables.numpy()
    _, h, w, off, nbytes, ncomp, hmax, vmax, ri, ioff = d[:10]
    mcus_x, mcus_y = -(-w // (8 * hmax)), -(-h // (8 * vmax))
    total = mcus_x * mcus_y
    n_int = -(-total // ri) if ri else 1
    starts = list(tables[ioff:ioff + 8 * n_int].view(np.int64)) + [nbytes]
    samp = [(hmax, vmax)] + [(1, 1)] * (ncomp - 1)
    coef = [np.zeros((mcus_y * v, mcus_x * hh, 64), np.int64) for hh, v in samp]
    dc_t = [_huff(tables, d[13 + c]) for c in range(ncomp)]
    ac_t = [_huff(tables, d[16 + c]) for c in range(ncomp)]
    mcu = 0
    for r in range(n_int):
        seg = data[off + starts[r]:off + starts[r + 1]]
        bits = np.unpackbits(seg)
        p = 0
        pred = [0] * ncomp
        for _ in range(min(ri, total - mcu) if ri else total):
            my, mx = divmod(mcu, mcus_x)
            for c in range(ncomp):
                hh, vv = samp[c]
                for v in range(vv):
                    for u in range(hh):
                        blk = coef[c][my * vv + v, mx * hh + u]
                        s, p = _decode_symbol(bits, p, dc_t[c])
                        diff, p = _receive(bits, p, s)
                        pred[c] += diff
                        blk[0] = (pred[c] + 32768) % 65536 - 32768              # JCOEF is int16
                        k = 1
                        while k < 64:
                            s, p = _decode_symbol(bits, p, ac_t[c])
                            run, size = s >> 4, s & 15
                            if size:
                                k += run
                                val, p = _receive(bits, p, size)
                                blk[NATURAL[k]] = val
                            elif run == 15:
                                k += 15
                            else:
                                break
                            k += 1
            mcu += 1
    return coef, (ncomp, hmax, vmax, mcus_x, mcus_y)


def range_limit(x):
    """libjpeg's post-IDCT range-limit table, indexed by x & 1023 (x centred on 0)."""
    v = np.asarray(x, np.int64) & 1023
    return np.where(v < 128, v + 128, np.where(v < 512, 255, np.where(v < 896, 0, v - 896))).astype(np.uint8)


def idct_islow(coef, q):
    """[..., 64] coefficients (natural order) x quant [64] -> [..., 8, 8] uint8 samples (jidctint.c jpeg_idct_islow)."""
    F = {k: int(v * 8192 + 0.5) for k, v in {"0_298": 0.298631336, "0_390": 0.390180644, "0_541": 0.541196100,
                                            "0_765": 0.765366865, "0_899": 0.899976223, "1_175": 1.175875602,
                                            "1_501": 1.501321110, "1_847": 1.847759065, "1_961": 1.961570560,
                                            "2_053": 2.053119869, "2_562": 2.562915447, "3_072": 3.072711026}.items()}
    x = (np.asarray(coef, np.int64) * np.asarray(q, np.int64)).reshape(coef.shape[:-1] + (8, 8))

    def one_d(v, pre, shift):
        # v[..., 8] along the last axis; pre: rounding folded into the even part (pass 2), shift: output descale
        z2, z3 = v[..., 2], v[..., 6]
        z1 = (z2 + z3) * F["0_541"]
        tmp2 = z1 + z3 * (-F["1_847"])
        tmp3 = z1 + z2 * F["0_765"]
        z2, z3 = v[..., 0] + pre, v[..., 4]
        tmp0, tmp1 = (z2 + z3) << 13, (z2 - z3) << 13
        tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
        t0, t1, t2, t3 = v[..., 7], v[..., 5], v[..., 3], v[..., 1]
        z1, z2, z3, z4 = t0 + t3, t1 + t2, t0 + t2, t1 + t3
        z5 = (z3 + z4) * F["1_175"]
        t0, t1, t2, t3 = t0 * F["0_298"], t1 * F["2_053"], t2 * F["3_072"], t3 * F["1_501"]
        z1, z2, z3, z4 = z1 * -F["0_899"], z2 * -F["2_562"], z3 * -F["1_961"] + z5, z4 * -F["0_390"] + z5
        t0, t1, t2, t3 = t0 + z1 + z3, t1 + z2 + z4, t2 + z2 + z3, t3 + z1 + z4
        out = [tmp10 + t3, tmp11 + t2, tmp12 + t1, tmp13 + t0, tmp13 - t0, tmp12 - t1, tmp11 - t2, tmp10 - t3]
        return np.stack([o >> shift for o in out], axis=-1)

    # pass 1: columns, DESCALE(x, CONST_BITS - PASS1_BITS) = (x + 2^10) >> 11
    cols = np.swapaxes(x, -1, -2)
    ws = one_d(cols + 0, 0, 0)
    ws = (ws + (1 << 10)) >> 11
    ws = np.swapaxes(ws, -1, -2)
    # pass 2: rows, rounding 2^(PASS1_BITS + 2) added to the DC term, >> (CONST_BITS + PASS1_BITS + 3)
    out = one_d(ws, 1 << 4, 18)
    return range_limit(out)


def planes(enc, i):
    coef, (ncomp, hmax, vmax, mx, my) = entropy_decode(enc, i)
    d = [int(v) for v in enc.desc[i]]
    tables = enc.tables.numpy()
    out = []
    for c in range(ncomp):
        q = tables[d[10 + c]:d[10 + c] + 128].view(np.uint16)
        s = idct_islow(coef[c], q)                              # [by, bx, 8, 8]
        by, bx = s.shape[:2]
        out.append(s.transpose(0, 2, 1, 3).reshape(by * 8, bx * 8))
    return out, (ncomp, hmax, vmax)


def _fancy_h(c, dw, out_w):
    c = c[:, :dw].astype(np.int64)
    left = np.concatenate([c[:, :1], c[:, :-1]], axis=1)
    right = np.concatenate([c[:, 1:], c[:, -1:]], axis=1)
    even = (3 * c + left + 1) >> 2
    odd = (3 * c + right + 2) >> 2
    even[:, 0], odd[:, -1] = c[:, 0], c[:, -1]
    return np.stack([even, odd], axis=2).reshape(c.shape[0], 2 * dw)[:, :out_w]


def _fancy_hv(c, dw, dh, out_w, out_h):
    c = c[:dh, :dw].astype(np.int64)
    above = np.concatenate([c[:1], c[:-1]], axis=0)
    below = np.concatenate([c[1:], c[-1:]], axis=0)
    rows = []
    for near in (above, below):                          # output rows 2i (row above) and 2i + 1 (row below)
        s = 3 * c + near
        left = np.concatenate([s[:, :1], s[:, :-1]], axis=1)
        right = np.concatenate([s[:, 1:], s[:, -1:]], axis=1)
        even = (3 * s + left + 8) >> 4
        odd = (3 * s + right + 7) >> 4
        even[:, 0] = (4 * s[:, 0] + 8) >> 4
        odd[:, -1] = (4 * s[:, -1] + 7) >> 4
        rows.append(np.stack([even, odd], axis=2).reshape(dh, 2 * dw))
    return np.stack(rows, axis=1).reshape(2 * dh, 2 * dw)[:out_h, :out_w]


def decode(enc, i):
    """Image i of an ``EncodedImages`` as ``Image.open(f).convert("RGB")`` gives it: uint8 [H, W, 3]."""
    d = [int(v) for v in enc.desc[i]]
    kind, h, w = d[:3]
    if kind == 1:
        return enc.data.numpy()[d[3]:d[3] + h * w * 3].reshape(h, w, 3).copy()
    p, (ncomp, hmax, vmax) = planes(enc, i)
    y = p[0][:h, :w].astype(np.int64)
    if ncomp == 1:
        return np.repeat(y[:, :, None], 3, axis=2).astype(np.uint8)
    dw, dh = -(-w // hmax), -(-h // vmax)
    ch = []
    for c in (1, 2):
        if (hmax, vmax) == (1, 1):
            ch.append(p[c][:h, :w].astype(np.int64))
        elif dw <= 2:                                            # libjpeg: no fancy upsampling this narrow
            ch.append(np.repeat(np.repeat(p[c], vmax, axis=0), hmax, axis=1)[:h, :w].astype(np.int64))
        elif vmax == 1:
            ch.append(_fancy_h(p[c][:h], dw, w))
        else:
            ch.append(_fancy_hv(p[c], dw, dh, w, h))
    cb, cr = ch[0] - 128, ch[1] - 128
    half = 1 << 15
    r = y + ((91881 * cr + half) >> 16)
    g = y + ((-22554 * cb + half - 46802 * cr) >> 16)
    b = y + ((116130 * cb + half) >> 16)
    return np.clip(np.stack([r, g, b], axis=2), 0, 255).astype(np.uint8)
