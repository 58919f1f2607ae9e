"""A progressive (SOF2) JPEG writer for tests: writes given quantised coefficients (oracle.decode_coefs order, as
jpeg_streams.write_baseline takes them) with any scan script, restart interval and Huffman tables. The entropy coding
restates jcphuff.c: the point transform of T.81 G.1.2 (DC shifted arithmetically, AC magnitudes shifted and then
signed), EOB runs up to 0x7FFF flushed at restart markers and at the end of a scan, and the correction bits of a
refinement scan buffered behind the EOB run or run symbol that precedes them. Its bytes need not be libjpeg's, only a
valid file. Plain Python, no GPU; test infrastructure only."""
import numpy as np

from jpeg_streams import JFIF_APP0, SAMPLING, _Bits, _codes, _seg, long_code_table, skewed_table

MAX_CORR_BITS = 1000   # jcphuff.c: correction bits buffered before an EOB run is forced out


# ---------------------------------------------------------------------------------------------------- scripts
def simple_script(ncomp=3):
    """jcparam.c jpeg_simple_progression."""
    if ncomp == 1:
        return [((0,), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((0,), 6, 63, 0, 2), ((0,), 1, 63, 2, 1), ((0,), 0, 0, 1, 0),
                ((0,), 1, 63, 1, 0)]
    return [((0, 1, 2), 0, 0, 0, 1), ((0,), 1, 5, 0, 2), ((2,), 1, 63, 0, 1), ((1,), 1, 63, 0, 1), ((0,), 6, 63, 0, 2),
            ((0,), 1, 63, 2, 1), ((0, 1, 2), 0, 0, 1, 0), ((2,), 1, 63, 1, 0), ((1,), 1, 63, 1, 0), ((0,), 1, 63, 1, 0)]


def _refined(comps, bands, al_first, dc=True):
    """DC interleaved over `comps` (when dc), first AC scans of every band at al_first, then one refinement pass per
    bit, band by band."""
    out = [(tuple(comps), 0, 0, 0, al_first)] if dc else []
    out += [((c,), ss, se, 0, al_first) for c in comps for ss, se in bands]
    for al in range(al_first - 1, -1, -1):
        if dc:
            out.append((tuple(comps), 0, 0, al + 1, al))
        out += [((c,), ss, se, al + 1, al) for c in comps for ss, se in bands]
    return out


def scripts(ncomp=3):
    """The catalogue of scan scripts, {name: script}. Every one sends every coefficient to its last bit."""
    comps = tuple(range(ncomp))
    per_comp_dc = [((c,), 0, 0, 0, 0) for c in comps]
    out = {
        "simple": simple_script(ncomp),
        # spectral selection only: every scan at Al = 0, DC in one scan per component
        "spectral": per_comp_dc + [((c,), ss, se, 0, 0) for c in comps for ss, se in ((1, 2), (3, 9), (10, 30), (31, 63))],
        # deep successive approximation: DC from Al = 3, AC first scans at Al = 3, three refinement passes per band
        "deep_sa": _refined(comps, ((1, 2), (3, 9), (10, 63)), 3),
        # refinement bands across bit 31/32 of the decoder's history mask, unlike the first scans' bands
        "cross32": [(comps, 0, 0, 0, 0)] + [((c,), ss, se, 0, 2) for c in comps for ss, se in ((1, 9), (10, 63))] +
                   [((c,), ss, se, 2, 1) for c in comps for ss, se in ((1, 31), (32, 63))] +
                   [((c,), ss, se, 1, 0) for c in comps for ss, se in ((1, 28), (29, 40), (41, 63))],
        # one scan per AC coefficient
        "per_coef": [(comps, 0, 0, 0, 0)] + [((c,), k, k, 0, 0) for k in range(1, 64) for c in comps],
        # Al up to 10: 10/11-bit magnitudes (an all-ones DQT) shifted far
        "al10": _refined(comps, ((1, 63),), 10),
        # high Al on low-amplitude content: EOB runs over (nearly) whole components
        "eob_long": _refined(comps, ((1, 63),), 5),
    }
    if ncomp == 3:
        # DC interleaved over Y and Cb, then Cr alone
        out["dc_ycb_cr"] = [((0, 1), 0, 0, 0, 1), ((2,), 0, 0, 0, 1)] + \
            [((c,), ss, se, 0, 0) for c in comps for ss, se in ((1, 5), (6, 63))] + \
            [((0, 1), 0, 0, 1, 0), ((2,), 0, 0, 1, 0)]
    return out


# ---------------------------------------------------------------------------------------------------- layout
class Layout:
    """Block geometry of a frame (oracle.geometry for three components; one block per MCU for one)."""

    def __init__(self, W, H, css, ncomp, oracle):
        if ncomp == 1:
            self.hs = self.vs = 1
            self.mcux, self.mcuy, self.bpm = -(-W // 8), -(-H // 8), 1
            self.wib, self.hib = [self.mcux], [self.mcuy]
        else:
            g = oracle.geometry(W, H, css)
            self.hs, self.vs = SAMPLING[css]
            self.mcux, self.mcuy, self.bpm = g.mcux, g.mcuy, g.bpm
            self.wib, self.hib = list(g.wib), list(g.hib)

    def comp_blocks(self, c):
        """Row indices of component c's own blocks in raster order (a non-interleaved scan's units)."""
        by, bx = np.meshgrid(np.arange(self.hib[c]), np.arange(self.wib[c]), indexing="ij")
        by, bx = by.ravel(), bx.ravel()
        if c:
            return (by * self.mcux + bx) * self.bpm + self.bpm - 3 + c
        my, mx = by // self.vs, bx // self.hs
        return (my * self.mcux + mx) * self.bpm + (by % self.vs) * self.hs + bx % self.hs

    def mcu_blocks(self, c):
        """Offsets in an MCU of component c's blocks."""
        return list(range(self.hs * self.vs)) if c == 0 else [self.bpm - 3 + c]


# ---------------------------------------------------------------------------------------------------- entropy coding
def _bitlen(v):
    return int(v).bit_length()


def _scan_ops(coef, lay, scan, ri):
    """The scan as a list of ops: (0, table, symbol), (1, value, nbits), (2,) a restart marker. table: index into the
    scan's component list."""
    comps, Ss, Se, Ah, Al = scan
    ops = []
    sym = lambda t, s: ops.append((0, t, s))
    bits = lambda v, n: ops.append((1, int(v), n)) if n else None
    if Ss == 0:
        if len(comps) > 1:
            nmcu = lay.mcux * lay.mcuy
            offs = [(i, b) for i, c in enumerate(comps) for b in lay.mcu_blocks(c)]
            units = [[(i, m * lay.bpm + b) for i, b in offs] for m in range(nmcu)]
        else:
            units = [[(0, int(b))] for b in lay.comp_blocks(comps[0])]
        dc = coef[:, 0].astype(np.int64) >> Al
        pred = [0] * len(comps)
        for u, unit in enumerate(units):
            if ri and u and u % ri == 0:
                ops.append((2,))
                pred = [0] * len(comps)
            for i, blk in unit:
                if Ah:
                    bits(dc[blk] & 1, 1)
                    continue
                d = int(dc[blk]) - pred[i]
                pred[i] = int(dc[blk])
                n = _bitlen(abs(d))
                sym(i, n)
                bits(d if d >= 0 else d - 1, n)
        return ops
    blocks = lay.comp_blocks(comps[0])
    band = coef[blocks, Ss:Se + 1].astype(np.int64)
    absv = np.abs(band) >> Al
    st = {"eobrun": 0, "be": []}

    def emit_eobrun():
        if st["eobrun"]:
            n = _bitlen(st["eobrun"]) - 1
            sym(0, n << 4)
            bits(st["eobrun"], n)
            st["eobrun"] = 0
            for b in st["be"]:
                bits(b, 1)
            st["be"] = []

    for u in range(len(blocks)):
        if ri and u and u % ri == 0:
            emit_eobrun()
            ops.append((2,))
        a, v = absv[u], band[u]
        nz = np.flatnonzero(a)
        if Ah == 0:                                  # encode_mcu_AC_first
            prev = -1
            for k in nz:
                r = k - prev - 1
                emit_eobrun()
                while r > 15:
                    sym(0, 0xF0)
                    r -= 16
                t = int(a[k])
                n = _bitlen(t)
                sym(0, (r << 4) | n)
                bits(t if v[k] > 0 else ~t, n)
                prev = k
            if prev < Se - Ss:
                st["eobrun"] += 1
                if st["eobrun"] == 0x7FFF:
                    emit_eobrun()
            continue
        ones = np.flatnonzero(a == 1)                 # encode_mcu_AC_refine
        eob = int(ones[-1]) if ones.size else -1
        prev, r, br = -1, 0, []
        for k in nz:
            r += k - prev - 1                         # zeros since the last symbol (correction positions do not count)
            prev = k
            while r > 15 and k <= eob:
                emit_eobrun()
                sym(0, 0xF0)
                r -= 16
                for b in br:
                    bits(b, 1)
                br = []
            t = int(a[k])
            if t > 1:                                 # already non-zero: a correction bit, buffered
                br.append(t & 1)
                continue
            emit_eobrun()
            sym(0, (r << 4) | 1)
            bits(0 if v[k] < 0 else 1, 1)
            for b in br:
                bits(b, 1)
            br, r = [], 0
        r += Se - Ss - prev
        if r > 0 or br:
            st["eobrun"] += 1
            st["be"] += br
            if st["eobrun"] == 0x7FFF or len(st["be"]) > MAX_CORR_BITS - 64 + 1:
                emit_eobrun()
    emit_eobrun()
    return ops


def _table(kind, freq, oracle):
    used = np.flatnonzero(freq)
    if kind == "optimal":
        bits, vals, n = oracle.gen_optimal_table(np.append(freq, 0).astype(np.uint32))
        return bits, vals[:n]
    if kind == "long":
        return long_code_table(used)
    if kind == "skewed":
        return skewed_table(freq, used)
    raise ValueError(kind)


def write_progressive(coef, qt, W, H, css, script, restart_interval=0, tables="optimal", ncomp=3, fill=0,
                      rotate_slots=False, eoi=True, oracle=None):
    """A progressive file of `coef` ((nblocks, 64) int16, zig-zag order, MCU by MCU: luma blocks then Cb, Cr; ncomp = 1:
    one block per MCU) with `script`, a list of (components, Ss, Se, Ah, Al).

    qt: (2, 64) natural-order tables (luma, chroma); restart_interval: MCUs (interleaved scans) or blocks (one
    component) per interval; tables: "optimal" (per scan, jpeg_gen_optimal_table), "long" (every code 11..16 bits) or
    "skewed" (a 1-bit code); fill: 0xFF bytes before every RSTn; rotate_slots: each scan's tables in other slots
    (0..3), so DHT redefines slots between scans; eoi: end with EOI."""
    lay = Layout(W, H, css, ncomp, oracle)
    coef = np.asarray(coef)
    hs, vs = (1, 1) if ncomp == 1 else SAMPLING[css]
    out = bytearray(b"\xff\xd8") + _seg(0xE0, JFIF_APP0)
    for slot in range(min(ncomp, 2)):
        out += _seg(0xDB, bytes([slot] + [int(qt[slot][z]) for z in _ZZ]))
    samp = [(hs << 4) | vs] + [0x11] * (ncomp - 1)
    out += _seg(0xC2, bytes([8]) + H.to_bytes(2, "big") + W.to_bytes(2, "big") + bytes([ncomp]) +
                b"".join(bytes([c + 1, samp[c], int(c > 0)]) for c in range(ncomp)))
    if restart_interval:
        out += _seg(0xDD, restart_interval.to_bytes(2, "big"))
    for si, scan in enumerate(script):
        comps, Ss, Se, Ah, Al = scan
        ops = _scan_ops(coef, lay, scan, restart_interval)
        cls = int(Ss > 0)
        # the scan's tables: one per component class (luma, chroma) it has, in slots 0/1 or rotated
        klass = [int(c > 0) for c in comps]
        slot = {k: (k + si) % 4 if rotate_slots else k for k in set(klass)}
        codes = {}
        if not (Ss == 0 and Ah):
            freq = {k: np.zeros(256, np.int64) for k in slot}
            for op in ops:
                if op[0] == 0:
                    freq[klass[op[1]]][op[2]] += 1
            dht = b""
            for k in sorted(slot):
                b, v = _table(tables, freq[k], oracle)
                codes[k] = _codes(b, v)
                dht += bytes([(cls << 4) | slot[k]]) + bytes(int(x) for x in b[1:17]) + bytes(int(x) for x in v)
            out += _seg(0xC4, dht)
        sel = [(slot[k] << 4 if cls == 0 and not Ah else slot[k]) if not (Ss == 0 and Ah) else 0 for k in klass]
        out += _seg(0xDA, bytes([len(comps)]) + b"".join(bytes([c + 1, s]) for c, s in zip(comps, sel)) +
                    bytes([Ss, Se, (Ah << 4) | Al]))
        w, rst = _Bits(), 0
        for op in ops:
            if op[0] == 0:
                w.put(*codes[klass[op[1]]][op[2]])
            elif op[0] == 1:
                w.put(op[1], op[2])
            else:
                w.flush()
                w.out += b"\xff" * fill + bytes([0xFF, 0xD0 + rst])
                rst = (rst + 1) & 7
        w.flush()
        out += w.out
    if eoi:
        out += b"\xff\xd9"
    return np.frombuffer(bytes(out), np.uint8).copy()


_ZZ = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
       28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
       47, 55, 62, 63]


# ---------------------------------------------------------------------------------------------------- incomplete files
def partial_coefs(coef, script, ncomp=3, oracle=None, lay=None):
    """The coefficients a decoder holds after `script` (a prefix of a complete one): each coefficient to the bits sent,
    zero where nothing was sent. A baseline file of these decodes to what libjpeg gives without block smoothing."""
    coef = np.asarray(coef, np.int64)
    out = np.zeros_like(coef)
    al = np.full((ncomp, 64), -1)
    for comps, Ss, Se, Ah, Al in script:
        for c in comps:
            al[c, Ss:Se + 1] = Al
    comp_of = np.zeros(coef.shape[0], np.int64)
    if ncomp == 3:
        bpm = lay.bpm
        comp_of = np.minimum(np.maximum(np.arange(coef.shape[0]) % bpm - (bpm - 3), 0), 2)
    for c in range(ncomp):
        rows = comp_of == c
        for k in range(64):
            a = al[c, k]
            if a < 0:
                continue
            v = coef[rows, k]
            out[rows, k] = (v >> a) << a if k == 0 else np.sign(v) * ((np.abs(v) >> a) << a)
    return out.astype(np.int16)


def smoothed(script, ncomp=3, gray_out=False, qt=None):
    """libjpeg-turbo's block-smoothing test (jdcoefct.c smoothing_ok) after `script`: every component's DC sent and some
    coefficient among zig-zag 1..9 of an output component unfinished (gray output: Y only)."""
    cb = np.full((ncomp, 10), -1)
    for comps, Ss, Se, Ah, Al in script:
        for c in comps:
            cb[c, Ss:min(Se, 9) + 1] = Al
    if (cb[:, 0] < 0).any():
        return False
    if qt is not None and any(int(qt[int(c > 0)][_ZZ[k]]) == 0 for c in range(ncomp) for k in range(10)):
        return False
    out = cb[:1] if gray_out else cb
    return bool((out[:, 1:] != 0).any())


def scan_segments(jpg):
    """[(start of the scan's DHT/SOS headers, end of its entropy-coded data)] of every scan, in file order."""
    b = bytes(jpg)
    p, out, head = 2, [], None
    while p + 1 < len(b):
        while b[p + 1] == 0xFF:
            p += 1
        m = b[p + 1]
        if m == 0xD9:
            break
        e = p + 2 + int.from_bytes(b[p + 2:p + 4], "big")
        if m == 0xC4 and head is None:
            head = p
        if m == 0xDA:
            while e + 1 < len(b) and not (b[e] == 0xFF and b[e + 1] not in (0, 0xFF) and not 0xD0 <= b[e + 1] <= 0xD7):
                e += 1
            if e + 1 >= len(b):
                e = len(b)
            out.append((p if head is None else head, e))
            head = None
        p = e
    return out


def cut(jpg, nbytes, eoi=True):
    """The first `nbytes` of a file, with EOI appended or not."""
    b = bytes(jpg)[:nbytes]
    return np.frombuffer(b + (b"\xff\xd9" if eoi else b""), np.uint8).copy()


# ---------------------------------------------------------------------------------------------------- the catalogue
GEOMETRIES = [(1, 1, 3), (17, 33, 3), (135, 121, 4), (257, 63, 1), (41, 58, 2), (37, 29, 0), (66, 35, 4)]
VARIANTS = [dict(), dict(restart_interval=3, tables="long", rotate_slots=True), dict(restart_interval=1, tables="skewed", fill=1),
            dict(restart_interval=7, fill=2, rotate_slots=True)]


def content(name):
    """(quality, synth amplitude) of a script's source: all-ones DQT and noise for al10, low amplitude for eob_long"""
    return {"al10": (100, 200), "eob_long": (90, 2)}.get(name, (90, 24))


def _source(oracle, W, H, css, quality, amp, seed, ncomp):
    """(coef, qt, W, H) of a synthetic image; one component: the luma blocks of a 4:4:4 file"""
    import jpeg_streams as J
    img = oracle.synth(W, H, seed, amp)
    coef, qt, W, H, _, _ = J.source(oracle.encode(img, 0 if ncomp == 1 else css, quality, 1), oracle)
    if ncomp == 1:
        coef, qt = np.ascontiguousarray(coef[0::3]), np.array([qt[0], qt[0]])
    return coef, qt, W, H


def entry(oracle, name, W, H, css, ncomp=3, seed=0, script=None, **kw):
    """(tag, file, script) of one catalogue entry"""
    q, amp = content(name)
    coef, qt, W, H = _source(oracle, W, H, css, q, amp, seed, ncomp)
    script = scripts(ncomp)[name] if script is None else script
    return coef, qt, W, H, script, write_progressive(coef, qt, W, H, css, script, oracle=oracle, ncomp=ncomp, **kw)


_CACHE = {}


def catalogue(oracle, big=True):
    """[(tag, file, ncomp)]: every script on ragged sizes and every subsampling, with restart intervals (in interleaved
    and non-interleaved scans), fill bytes, long-code / skewed / per-scan optimal tables and DHT in rotated slots, in
    colour and one-component files; 640x360 files, and files of about 2 MP with and without restart intervals."""
    key = ("catalogue", big)
    if key in _CACHE:
        return _CACHE[key]
    out = []
    for ncomp in (3, 1):
        for si, name in enumerate(scripts(ncomp)):
            for gi in range(3):
                W, H, css = GEOMETRIES[(si + 2 * gi) % len(GEOMETRIES)]
                kw = VARIANTS[(si + gi) % len(VARIANTS)]
                *_, jpg = entry(oracle, name, W, H, css, ncomp, seed=si * 3 + gi, **kw)
                out.append((f"{name}/{ncomp}c/{W}x{H}/css{css if ncomp == 3 else 'gray'}/{kw}", jpg, ncomp))
    for name, css, kw in (("simple", 3, {}), ("deep_sa", 1, dict(restart_interval=5)), ("cross32", 4, dict(restart_interval=40))):
        *_, jpg = entry(oracle, name, 640, 360, css, seed=7, **kw)
        out.append((f"{name}/3c/640x360/css{css}/{kw}", jpg, 3))
    if big:
        *_, jpg = entry(oracle, "simple", 1920, 1080, 3, seed=9)
        out.append(("simple/3c/1920x1080/css3/no restarts", jpg, 3))
        # 256 x 136 blocks per component: EOB runs reach 0x7FFF, the first one exactly at the restart boundary
        *_, jpg = entry(oracle, "eob_long", 2048, 1088, 0, seed=10, restart_interval=0x7FFF)
        out.append(("eob_long/3c/2048x1088/css0/ri 32767", jpg, 3))
        *_, jpg = entry(oracle, "cross32", 1920, 1088, 1, seed=11, restart_interval=97)
        out.append(("cross32/3c/1920x1088/css1/ri 97", jpg, 3))
    _CACHE[key] = out
    return out


def incomplete(oracle):
    """[(tag, file, ncomp, script_received)] of incomplete progressive files: catalogue-style files cut after each scan
    (with and without EOI), cut inside their last and an earlier scan, next to a restart marker, and scripts that stop
    short (no final refinement, no chroma AC, only zig-zag 10.. unfinished, only the DC refinement missing).
    script_received: the scans a decoder has started, which decide block smoothing."""
    if "incomplete" in _CACHE:
        return _CACHE["incomplete"]
    comps = (0, 1, 2)
    short = {
        "no_final_refinement": simple_script()[:-1],
        "no_chroma_ac": [(comps, 0, 0, 0, 0), ((0,), 1, 63, 0, 0)],
        "only_10_63_unfinished": [(comps, 0, 0, 0, 0)] + [((c,), 1, 9, 0, 0) for c in comps] + [((c,), 10, 63, 0, 1) for c in comps],
        "only_dc_refinement_missing": [(comps, 0, 0, 0, 1)] + [((c,), 1, 63, 0, 0) for c in comps],
        "y_zz9_unfinished": [(comps, 0, 0, 0, 0)] + [((c,), 1, 63, 0, 0) for c in (1, 2)] + [((0,), 1, 8, 0, 0), ((0,), 9, 63, 0, 1)],
    }
    out = []
    for name, script in short.items():
        *_, jpg = entry(oracle, "simple", 57, 41, 3, seed=3, script=script)
        out.append((f"short/{name}", jpg, 3, script))
    bases = [("simple", 3, 135, 121, 3, {}), ("deep_sa", 3, 67, 45, 4, dict(restart_interval=5)),
             ("simple", 1, 57, 41, 0, dict(restart_interval=3)), ("cross32", 3, 41, 58, 1, dict(restart_interval=2, fill=1))]
    for name, ncomp, W, H, css, kw in bases:
        *_, script, jpg = entry(oracle, name, W, H, css, ncomp, seed=5, **kw)
        segs = scan_segments(jpg)
        tag = f"{name}/{ncomp}c/{W}x{H}/css{css}/{kw}"
        for k in range(1, len(segs)):
            for eoi in (True, False):
                out.append((f"{tag}/after scan {k}/eoi {eoi}", cut(jpg, segs[k - 1][1], eoi), ncomp, script[:k]))
        for k in (len(segs) - 1, 1):   # inside the last scan, and inside the second
            s0, e0 = segs[k]
            data0 = bytes(jpg).index(b"\xff\xda", s0) + 2 + int.from_bytes(bytes(jpg)[bytes(jpg).index(b"\xff\xda", s0) + 2:][:2], "big")
            cuts = {"first byte": data0 + 1, "middle": (data0 + e0) // 2, "last byte": e0 - 1}
            seg = bytes(jpg)[data0:e0]
            rst = [data0 + i for i in range(len(seg) - 1) if seg[i] == 0xFF and 0xD0 <= seg[i + 1] <= 0xD7]
            if rst:
                r = rst[len(rst) // 2]
                cuts.update({"before RSTn": r, "after RSTn": r + 2})
            for where, n in cuts.items():
                for eoi in (True, False):
                    out.append((f"{tag}/inside scan {k + 1} ({where})/eoi {eoi}", cut(jpg, n, eoi), ncomp, script[:k + 1]))
    _CACHE["incomplete"] = out
    return out
