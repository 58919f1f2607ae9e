"""A baseline JPEG writer for tests: re-writes the quantised coefficients of an existing stream (oracle.decode_coefs) in
the layouts other writers use (table slots, component ids, SOF1 and 16-bit DQT, restart intervals of any length, fill
bytes, split or moved table segments, APPn/COM segments, JFIF / Adobe markers) and with other Huffman tables (long
codes, a 1-bit code). The coefficients and quantisation values are the source's, so every stream it writes decodes in
libjpeg to the source's pixels, whatever its layout. Plain Python, no GPU; test infrastructure only."""
import numpy as np

# zigzag position -> natural (row-major) index
ZZ = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
      28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
      47, 55, 62, 63]

SAMPLING = {0: (1, 1), 1: (2, 1), 2: (1, 2), 3: (2, 2), 4: (4, 1)}   # css -> luma (h, v)


# ---------------------------------------------------------------------------------------------------- tables
def std_huff(oracle):
    """The standard tables (T.81 K.3) as {(class, slot): (bits[17], vals)}: DC0, AC0, DC1, AC1."""
    bits, vals = oracle.std_tables()
    out = {}
    for t, key in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))):
        n = int(bits[t][1:].sum())
        out[key] = (np.array(bits[t], np.uint8), np.array(vals[t][:n], np.uint8))
    return out


def _canonical(lengths):
    """{symbol: length} -> (bits, vals) in canonical order (by length, then symbol)."""
    bits = np.zeros(17, np.uint8)
    for l in lengths.values():
        bits[l] += 1
    vals = np.array(sorted(lengths, key=lambda s: (lengths[s], s)), np.uint8)
    _check_kraft(bits)
    return bits, vals


def _check_kraft(bits):
    code = 0
    for l in range(1, 17):
        code += int(bits[l])
        assert code <= (1 << l) - (1 if l == 16 else 0), "over-full table (the all-ones code stays reserved)"
        code <<= 1
    # no all-ones code of any length: the last code of the longest length is below all ones
    lmax = max(l for l in range(1, 17) if bits[l])
    total = sum(int(bits[l]) << (lmax - l) for l in range(1, lmax + 1))
    assert total < (1 << lmax), "all-ones code used"


def long_code_table(symbols):
    """Every symbol gets a code of 11..16 bits (round robin over the lengths), so that none is in a 10-bit lookup."""
    symbols = sorted(set(int(s) for s in symbols))
    return _canonical({s: 11 + i % 6 for i, s in enumerate(symbols)})


def skewed_table(freq, symbols):
    """The most frequent of `symbols` gets a 1-bit code, every other one the shortest equal length that fits."""
    freq = np.asarray(freq)
    used = sorted(set(int(s) for s in symbols), key=lambda s: -int(freq[s]))
    rest = used[1:]
    l = 2
    while (1 << (l - 1)) - 1 < len(rest):
        l += 1
    lengths = {used[0]: 1}
    lengths.update({s: l for s in rest})
    return _canonical(lengths)


# ---------------------------------------------------------------------------------------------------- entropy coding
def _codes(bits, vals):
    out, code, k = {}, 0, 0
    for l in range(1, 17):
        for _ in range(int(bits[l])):
            out[int(vals[k])] = (code, l)
            code += 1
            k += 1
        code <<= 1
    return out


class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, v, n):
        self.acc = (self.acc << n) | (v & ((1 << n) - 1))
        self.n += n
        while self.n >= 8:
            self.n -= 8
            b = (self.acc >> self.n) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)
        self.acc &= (1 << self.n) - 1

    def flush(self):   # pad with 1-bits
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def _nbits(v):
    return int(abs(int(v))).bit_length()


def entropy_segment(coef, nblk_per_comp, dc, ac, restart_interval=0, fill=0):
    """coef: (nmcu * bpm, 64) int16, zigzag order, blocks of an MCU component by component (nblk_per_comp of them).
    dc/ac: per component {symbol: (code, length)}. Returns the stuffed bytes with RSTn markers (fill 0xFF before each)."""
    bpm = sum(nblk_per_comp)
    comp = [c for c, k in enumerate(nblk_per_comp) for _ in range(k)]
    nmcu = coef.shape[0] // bpm
    w = _Bits()
    pred = [0] * len(nblk_per_comp)
    rst = 0
    c64 = coef.astype(np.int64)
    for m in range(nmcu):
        if restart_interval and m and m % restart_interval == 0:
            w.flush()
            w.out += b"\xff" * fill + bytes([0xFF, 0xD0 + rst])
            rst = (rst + 1) & 7
            pred = [0] * len(nblk_per_comp)
        for b in range(bpm):
            c = comp[b]
            blk = c64[m * bpm + b]
            d = int(blk[0]) - pred[c]
            pred[c] = int(blk[0])
            s = _nbits(d)
            w.put(*dc[c][s])
            if s:
                w.put(d if d >= 0 else d - 1, s)
            run = 0
            nz = np.nonzero(blk[1:])[0]
            last = int(nz[-1]) + 1 if nz.size else 0
            for k in range(1, last + 1):
                v = int(blk[k])
                if v == 0:
                    run += 1
                    continue
                while run > 15:
                    w.put(*ac[c][0xF0])
                    run -= 16
                s = _nbits(v)
                w.put(*ac[c][(run << 4) | s])
                w.put(v if v >= 0 else v - 1, s)
                run = 0
            if last < 63:
                w.put(*ac[c][0x00])
    w.flush()
    return bytes(w.out)


# ---------------------------------------------------------------------------------------------------- the writer
def _seg(marker, payload, fill=0):
    return b"\xff" * fill + bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)


JFIF_APP0 = b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00"


def adobe_app14(transform):
    return b"Adobe" + bytes([0, 100, 0, 0, 0, 0, transform])


def write_baseline(coef, qt, W, H, css, *, ncomp=3, htabs=None, hsel=((0, 0), (1, 1), (1, 1)), qtabs=None,
                   qsel=(0, 1, 1), ids=(1, 2, 3), sof=0xC0, dqt16=False, restart_interval=0, fill=0,
                   one_segment=False, tables_after_sof=False, segments=(), late_segments=(), jfif=True, adobe=None,
                   oracle=None):
    """A baseline stream of `coef` (oracle.decode_coefs order: MCU by MCU, luma blocks then Cb, Cr; zigzag order).

    qt: (2, 64) natural-order tables of the source (luma, chroma); qtabs {slot: 64 natural-order values} overrides them.
    htabs {(class, slot): (bits, vals)}: the tables written (default: the standard ones); hsel: (DC slot, AC slot) per
    component; qsel: quantisation slot per component; ids: component ids; sof: 0xC0 / 0xC1; dqt16: 16-bit DQT entries;
    restart_interval: MCUs per interval (0: none); fill: 0xFF bytes before every marker after SOI; one_segment: all
    DQT tables in one segment and all DHT tables in one; tables_after_sof: DQT/DHT between SOF and SOS;
    segments / late_segments: (marker, payload) right after SOI's APP0/APP14 / right before SOS; jfif: a JFIF APP0;
    adobe: None or the transform of an Adobe APP14. ncomp = 1: `coef` holds one component, one block per MCU."""
    if htabs is None:
        htabs = std_huff(oracle)
    if qtabs is None:
        qtabs = {0: qt[0], 1: qt[1]}
    hs, vs = (1, 1) if ncomp == 1 else SAMPLING[css]
    used_q = sorted(set(qsel[:ncomp]))
    used_h = sorted(set([(0, hsel[c][0]) for c in range(ncomp)] + [(1, hsel[c][1]) for c in range(ncomp)]))

    def dqt_payload(slot):
        v = [int(qtabs[slot][ZZ[k]]) for k in range(64)]
        if dqt16:
            return bytes([0x10 | slot]) + b"".join(x.to_bytes(2, "big") for x in v)
        assert max(v) <= 255
        return bytes([slot] + v)

    def dht_payload(key):
        bits, vals = htabs[key]
        return bytes([(key[0] << 4) | key[1]]) + bytes(int(b) for b in bits[1:17]) + bytes(int(v) for v in vals)

    if one_segment:
        tables = _seg(0xDB, b"".join(dqt_payload(s) for s in used_q), fill) + \
            _seg(0xC4, b"".join(dht_payload(k) for k in used_h), fill)
    else:
        tables = b"".join(_seg(0xDB, dqt_payload(s), fill) for s in used_q) + \
            b"".join(_seg(0xC4, dht_payload(k), fill) for k in used_h)
    samp = [(hs << 4) | vs] + [0x11] * (ncomp - 1)
    frame = bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([ncomp]) + \
        b"".join(bytes([ids[c], samp[c], qsel[c]]) for c in range(ncomp))
    out = bytearray(b"\xff\xd8")
    if jfif:
        out += _seg(0xE0, JFIF_APP0, fill)
    if adobe is not None:
        out += _seg(0xEE, adobe_app14(adobe), fill)
    for m, p in segments:
        out += _seg(m, p, fill)
    if not tables_after_sof:
        out += tables
    out += _seg(sof, frame, fill)
    if tables_after_sof:
        out += tables
    for m, p in late_segments:
        out += _seg(m, p, fill)
    if restart_interval:
        out += _seg(0xDD, restart_interval.to_bytes(2, "big"), fill)
    out += _seg(0xDA, bytes([ncomp]) + b"".join(bytes([ids[c], (hsel[c][0] << 4) | hsel[c][1]]) for c in range(ncomp))
                + bytes([0, 63, 0]), fill)
    nblk = [1] if ncomp == 1 else [hs * vs, 1, 1]
    dc = [_codes(*htabs[(0, hsel[c][0])]) for c in range(ncomp)]
    ac = [_codes(*htabs[(1, hsel[c][1])]) for c in range(ncomp)]
    out += entropy_segment(coef, nblk, dc, ac, restart_interval, fill)
    out += b"\xff" * fill + b"\xff\xd9"
    return np.frombuffer(bytes(out), np.uint8).copy()


def source(jpg, oracle):
    """(coef, qt, W, H, css, restart_interval) of a baseline stream, as write_baseline takes them."""
    coef, info = oracle.decode_coefs(jpg)
    qt = np.array(info.qt, np.uint16)
    return coef, qt, info.W, info.H, info.css, info.restart_interval


# ---------------------------------------------------------------------------------------------------- byte rewrites
def _scan_start(jpg):
    b = bytes(jpg)
    p = 2
    while True:
        while b[p + 1] == 0xFF:
            p += 1
        m = b[p + 1]
        L = int.from_bytes(b[p + 2:p + 4], "big")
        p += 2 + L
        if m == 0xDA:
            return p


def insert_fill(jpg, n):
    """n fill bytes (0xFF) before every RSTn and before EOI of a one-scan stream."""
    b = bytes(jpg)
    p = _scan_start(b)
    out = bytearray(b[:p])
    i = p
    while i < len(b):
        if b[i] == 0xFF and i + 1 < len(b) and (0xD0 <= b[i + 1] <= 0xD7 or b[i + 1] == 0xD9):
            out += b"\xff" * n
            out += b[i:i + 2]
            i += 2
            continue
        out.append(b[i])
        i += 1
    return np.frombuffer(bytes(out), np.uint8).copy()


def drop_eoi(jpg):
    b = bytes(jpg)
    assert b[-2:] == b"\xff\xd9"
    return np.frombuffer(b[:-2], np.uint8).copy()


def append_after_eoi(jpg, data):
    return np.frombuffer(bytes(jpg) + bytes(data), np.uint8).copy()


def add_dri0(jpg):
    """A DRI segment with interval 0 right after SOI (any later DRI still counts)."""
    b = bytes(jpg)
    return np.frombuffer(b[:2] + _seg(0xDD, b"\x00\x00") + b[2:], np.uint8).copy()


def _segments(b):
    """(marker, start, end) of every marker after SOI (fill bytes skipped; a scan's entropy data ends its segment)."""
    p, out = 2, []
    while p + 1 < len(b):
        while p + 1 < len(b) and b[p + 1] == 0xFF:
            p += 1
        m = b[p + 1]
        if m == 0xD9:
            out.append((m, p, p + 2))
            break
        e = p + 2 + int.from_bytes(b[p + 2:p + 4], "big")
        if m == 0xDA:
            while e + 1 < len(b) and not (b[e] == 0xFF and b[e + 1] != 0 and not 0xD0 <= b[e + 1] <= 0xD7):
                e += 1
        out.append((m, p, e))
        p = e
    return out


def restyle(jpg, ids=None, drop_jfif=False, adobe=None, tq=None):
    """The same stream (baseline or progressive) with other component ids (SOF and every SOS), without its JFIF APP0,
    with an Adobe APP14 (transform `adobe`) after SOI, or with other quantisation slot numbers in SOF."""
    b = bytes(jpg)
    segs = _segments(b)
    out = bytearray(b[:2])
    if adobe is not None:
        out += _seg(0xEE, adobe_app14(adobe))
    old_ids = None
    for i, (m, s, _) in enumerate(segs):
        chunk = bytearray(b[s:segs[i + 1][1] if i + 1 < len(segs) else len(b)])
        if m == 0xE0 and drop_jfif and chunk[4:9] == b"JFIF\x00":
            continue
        if m in (0xC0, 0xC1, 0xC2):
            old_ids = [chunk[10 + 3 * c] for c in range(chunk[9])]
            for c in range(chunk[9]):
                if ids is not None:
                    chunk[10 + 3 * c] = ids[c]
                if tq is not None:
                    chunk[12 + 3 * c] = tq[c]
        if m == 0xDA and ids is not None:
            for k in range(chunk[4]):
                chunk[5 + 2 * k] = ids[old_ids.index(chunk[5 + 2 * k])]
        out += chunk
    return np.frombuffer(bytes(out), np.uint8).copy()


def write_noninterleaved(coef, qt, W, H, oracle):
    """A 4:4:4 baseline stream with one scan per component (legal, and decoded by libjpeg)."""
    h = std_huff(oracle)
    one = [write_baseline(np.ascontiguousarray(coef[c::3]), qt, W, H, 0, ncomp=1, htabs=h, hsel=((c > 0, c > 0),) * 3,
                          qsel=(int(c > 0),) * 3, ids=(c + 1,) * 3, oracle=oracle).tobytes() for c in range(3)]
    head = write_baseline(coef, qt, W, H, 0, oracle=oracle).tobytes()
    sos = [s for m, s, _ in _segments(head) if m == 0xDA][0]
    out = bytearray(head[:sos])
    for c in range(3):
        s = [s for m, s, _ in _segments(one[c]) if m == 0xDA][0]
        out += one[c][s:-2]
    out += b"\xff\xd9"
    return np.frombuffer(bytes(out), np.uint8).copy()


# ---------------------------------------------------------------------------------------------------- the corpus
SIZES = {0: (37, 29), 1: (50, 33), 2: (41, 58), 3: (67, 45), 4: (75, 20)}


def _entry(name, jpg, accept, src=None, progressive=False):
    return {"name": name, "jpg": np.asarray(jpg, np.uint8), "accept": accept,
            "ref": np.asarray(jpg if src is None else src, np.uint8), "progressive": progressive}


def writer_streams(oracle, css, quality=90, size=None):
    """(name, stream) of every writer layout for one source; every one holds the source's coefficients and tables."""
    W, H = size or SIZES[css]
    img = oracle.synth(W, H, 11 * css + quality, 24)
    src = oracle.encode(img, css, quality, 1)
    coef, qt, W, H, _, _ = source(src, oracle)
    g = oracle.geometry(W, H, css)
    h = std_huff(oracle)
    hist = oracle.histogram(coef, g.bpm)
    # every symbol of the standard tables (restart intervals change the DC differences) gets a code
    keys = ((0, 0), (1, 0), (0, 1), (1, 1))   # DC0, AC0, DC1, AC1: the order of oracle.histogram
    long = {k: long_code_table(h[k][1]) for k in keys}
    skew = {k: skewed_table(hist[t], h[k][1]) for t, k in enumerate(keys)}
    junk = b"\xff\xd9 \xff\xc0 \xff\xda \xff\xff\x00"
    out = [("plain", src),
           ("sof1_dqt16", dict(sof=0xC1, dqt16=True)),
           ("dqt16", dict(dqt16=True)),
           ("slots23", dict(htabs={(0, 3): h[(0, 0)], (1, 2): h[(1, 0)], (0, 2): h[(0, 1)], (1, 3): h[(1, 1)]},
                            hsel=((3, 2), (2, 3), (2, 3)), qtabs={3: qt[0], 2: qt[1]}, qsel=(3, 2, 2))),
           ("shared_huff", dict(htabs={(0, 0): h[(0, 0)], (1, 0): h[(1, 0)]}, hsel=((0, 0),) * 3)),
           ("ids_jfif_rgb", dict(ids=(82, 71, 66))),
           ("ids_jfif_012", dict(ids=(0, 1, 2))),
           ("adobe1_rgb_ids", dict(jfif=False, adobe=1, ids=(82, 71, 66))),
           ("no_markers_ids_012", dict(jfif=False, ids=(0, 1, 2))),
           ("fill2_every_marker", dict(fill=2, restart_interval=3)),
           ("app_com_before_sos", dict(segments=[(0xFE, junk), (0xE2, junk)], late_segments=[(0xE1, junk), (0xFE, b"")])),
           ("one_segment_after_sof", dict(one_segment=True, tables_after_sof=True)),
           ("tables_after_sof", dict(tables_after_sof=True)),
           ("ri1", dict(restart_interval=1)),
           ("ri7", dict(restart_interval=7)),
           ("ri_row_plus_1", dict(restart_interval=g.mcux + 1)),
           ("long_codes", dict(htabs=long)),
           ("long_codes_ri5", dict(htabs=long, restart_interval=5)),
           ("skewed", dict(htabs=skew)),
           ("skewed_shared_fill1", dict(htabs=skew, restart_interval=2, fill=1))]
    res = []
    for name, v in out:
        res.append((name, v if not isinstance(v, dict) else write_baseline(coef, qt, W, H, css, oracle=oracle, **v)))
    rsrc = oracle.encode(img, css, quality, 1, 3)
    for n in (1, 2, 5):
        res.append((f"fill{n}_rst_eoi", insert_fill(rsrc, n)))
    res.append(("fill2_eoi", insert_fill(src, 2)))
    res.append(("no_eoi", drop_eoi(src)))
    res.append(("no_eoi_rst", drop_eoi(rsrc)))
    res.append(("after_eoi", append_after_eoi(src, b"\x00\xff\xd9\xff\xd8tail")))
    res.append(("dri0", add_dri0(src)))
    return src, res


def corpus(oracle, with_pillow=True):
    """Every interop stream with the product's verdict: accept (GPU pixels = cv2's of `ref`) or refuse (B2J_EFORMAT)."""
    out = []
    for css in range(5):
        src, streams = writer_streams(oracle, css)
        for name, jpg in streams:
            out.append(_entry(f"{css}/{name}", jpg, True, src))
        coef, qt, W, H, _, _ = source(src, oracle)
        out.append(_entry(f"{css}/adobe0", write_baseline(coef, qt, W, H, css, oracle=oracle, jfif=False, adobe=0), False))
        out.append(_entry(f"{css}/adobe0_ids_rgb", write_baseline(coef, qt, W, H, css, oracle=oracle, jfif=False, adobe=0,
                                                                 ids=(82, 71, 66)), False))
        out.append(_entry(f"{css}/ids_rgb_no_markers", restyle(src, ids=(82, 71, 66), drop_jfif=True), False))
        out.append(_entry(f"{css}/tq_4_5", restyle(src, tq=(4, 5, 5)), False))
        out.append(_entry(f"{css}/separate_cr_qt", write_baseline(coef, qt, W, H, css, oracle=oracle, qtabs={0: qt[0], 1: qt[1], 2: qt[1]},
                                                                qsel=(0, 1, 2)), False))
        W, H = SIZES[css]
        prog = oracle.encode_progressive(oracle.synth(W, H, css, 24), css, 90)
        out.append(_entry(f"{css}/prog", prog, True, progressive=True))
        out.append(_entry(f"{css}/prog_adobe1", restyle(prog, drop_jfif=True, adobe=1), True, prog, progressive=True))
        out.append(_entry(f"{css}/prog_adobe0", restyle(prog, drop_jfif=True, adobe=0), False, progressive=True))
        out.append(_entry(f"{css}/prog_ids_rgb", restyle(prog, ids=(82, 71, 66), drop_jfif=True), False, progressive=True))
        out.append(_entry(f"{css}/prog_tq_4_5", restyle(prog, tq=(4, 5, 5)), False, progressive=True))
    src, _ = writer_streams(oracle, 0, 100)
    coef, qt, W, H, _, _ = source(src, oracle)
    assert np.array_equal(qt[0], qt[1])
    out.append(_entry("0/one_qt_q100", write_baseline(coef, qt, W, H, 0, oracle=oracle, qsel=(0, 0, 0)), True, src))
    out.append(_entry("0/noninterleaved", write_noninterleaved(coef, qt, W, H, oracle), False))
    if with_pillow:
        out += pillow_corpus(oracle)
    return out


def pillow_corpus(oracle):
    """Streams Pillow's libjpeg writer makes with the options cameras and libraries use; [] without Pillow."""
    try:
        from PIL import Image
    except ImportError:
        return []
    import io
    W, H = 61, 43
    rgb = Image.fromarray(np.ascontiguousarray(oracle.synth(W, H, 5, 24)[:, :, ::-1]))
    t1 = [1 + (k * 7) % 90 for k in range(64)]
    t2 = [2 + (k * 5) % 120 for k in range(64)]
    big = [200 + k * 9 for k in range(64)]   # > 255: 16-bit DQT, SOF1
    ff = b"\xff\xd9\xff\xc0\xff\xda\xff"
    icc = bytes(range(256)) * 3
    exif = b"Exif\x00\x00MM\x00*\x00\x00\x00\x08\x00\x00" + ff
    v = [("ss0", dict(subsampling=0), True), ("ss1", dict(subsampling=1), True), ("ss2", dict(subsampling=2), True),
         ("ss0_opt", dict(subsampling=0, optimize=True), True), ("ss2_opt", dict(subsampling=2, optimize=True), True),
         ("q_one_table", dict(qtables=[t1]), True), ("q_two_tables", dict(qtables=[t1, t2]), True),
         ("q_16bit", dict(qtables=[big, t2]), True), ("q_16bit_both", dict(qtables=[big, big], subsampling=0), True),
         ("q_three_tables", dict(qtables=[t1, t2, t1]), False),
         ("rst_rows", dict(restart_marker_rows=1), True), ("rst_blocks5", dict(restart_marker_blocks=5), True),
         ("rst_blocks5_ss0", dict(restart_marker_blocks=5, subsampling=0), True),
         ("comment", dict(comment=ff), True), ("exif", dict(exif=exif), True), ("icc", dict(icc_profile=icc), True),
         ("progressive", dict(progressive=True), True), ("progressive_16bit", dict(progressive=True, qtables=[big, t2]), True),
         ("keep_rgb", dict(subsampling=0, keep_rgb=True), False),
         ("keep_rgb_progressive", dict(subsampling=0, keep_rgb=True, progressive=True), False)]
    out = []
    for name, kw, accept in v:
        b = io.BytesIO()
        rgb.save(b, "JPEG", **(kw if "qtables" in kw else dict(kw, quality=85)))   # a quality would scale qtables
        j = np.frombuffer(b.getvalue(), np.uint8).copy()
        out.append(_entry("pillow/" + name, j, accept, progressive=bool(kw.get("progressive"))))
    return out
