"""Randomised parity run against the checker (development aid, needs a B200): random sizes up to 2000 x 1500, all
samplings, qualities, both Huffman modes; every encode also with the entropy coder's small-buffer recovery path
(debug flag 2), with restart rows now and then, and every stream decoded back and compared with the checker's decode.
    python scripts/dev/stress.py [cases] [seed]"""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
import nvjpeg_imagecompressor_b200 as P
import oracle as O
ncase = int(sys.argv[1]) if len(sys.argv) > 1 else 150
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 7)
CAPW, CAPH = 2000, 1500
engs = {}
nfail = ntot = 0
t0 = time.time()
for case in range(ncase):
    css = int(rng.integers(0, 5)); q = int(rng.choice([30, 60, 75, 90, 95, 98, 100])); opt = int(rng.integers(0, 2))
    small = rng.random() < 0.5
    W = int(rng.integers(1, 200 if small else CAPW)); H = int(rng.integers(1, 200 if small else CAPH))
    kind = rng.random()
    if kind < 0.6: img = O.synth(W, H, case, int(rng.choice([0, 2, 8, 40])))
    elif kind < 0.8: img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    else: img = np.full((H, W, 3), int(rng.integers(0, 256)), np.uint8)
    key = (css, q, opt)
    if key not in engs: engs[key] = P.Engine(CAPW, CAPH, q, bool(opt), css)
    eng = engs[key]
    g = O.geometry(W, H, css)
    rows = int(rng.integers(1, 4)) if rng.random() < 0.25 and rng.integers(1, 4) * g.mcux <= 65535 else 0
    want = O.encode(img, css, q, opt, rows * g.mcux) if rows else O.encode(img, css, q, opt)
    for dbg in ((0,) if rows else (0, 2)):
        eng.set_debug(dbg); eng.set_restart_rows(rows)
        jpg = eng.encode(img)
        ntot += 1
        if not (jpg.size == want.size and np.array_equal(jpg, want)):
            nfail += 1
            print(f"ENCODE FAIL case{case} css{css} q{q} opt{opt} {W}x{H} rows{rows} dbg{dbg} len {jpg.size}/{want.size}")
    eng.set_debug(0); eng.set_restart_rows(0)
    dec = eng.decode(want)
    ntot += 1
    if not np.array_equal(dec, O.decode(want)):
        nfail += 1
        print(f"DECODE FAIL case{case} css{css} q{q} opt{opt} {W}x{H} rows{rows}")
print({"checks": ntot, "fail": nfail, "seconds": round(time.time() - t0, 1)})
sys.exit(1 if nfail else 0)
