"""Progressive (SOF2) files with any scan script on the CPU (tests/prog_streams.py): the writer's own check against live
cv2, the CPU checkers against cv2 on every file of the catalogue, and incomplete files (cut after or inside a scan,
scripts that stop short). libjpeg-turbo block-smooths a file that leaves low-frequency coefficients unfinished; the
rule for when it does is pinned to live cv2 here, and the checkers refuse such files as the product does.
tests/test_gpu_prog_streams.py decodes the same files on the GPU."""
import cv2
import numpy as np
import pytest

import oracle as O
import jpeg_streams as J
import prog_streams as PS


def dec(jpg, flag=cv2.IMREAD_COLOR):
    out = cv2.imdecode(np.asarray(jpg, np.uint8), flag)
    assert out is not None
    return out


def with_eoi(jpg):
    """libjpeg decodes a file that ends without EOI as if it had one (with a warning, which cv2 turns into a refusal)"""
    b = bytes(jpg)
    return jpg if b.endswith(b"\xff\xd9") else np.frombuffer(b + b"\xff\xd9", np.uint8)


@pytest.mark.parametrize("ncomp", (3, 1))
def test_writer_matches_baseline(oracle, ncomp):
    """every script, size, restart interval and table kind: the progressive file decodes in cv2 to the pixels of a
    baseline file of the same coefficients"""
    h = J.std_huff(oracle)
    n = 0
    for si, name in enumerate(PS.scripts(ncomp)):
        for gi in range(len(PS.GEOMETRIES)):
            W, H, css = PS.GEOMETRIES[gi]
            kw = PS.VARIANTS[(si + gi) % len(PS.VARIANTS)]
            if name == "per_coef" and W * H > 5000:
                continue
            coef, qt, W, H, script, jpg = PS.entry(oracle, name, W, H, css, ncomp, seed=gi, **kw)
            base = J.write_baseline(coef, qt, W, H, css, ncomp=ncomp, htabs=h, oracle=oracle)
            flag = cv2.IMREAD_COLOR if ncomp == 3 else cv2.IMREAD_UNCHANGED
            assert np.array_equal(dec(jpg, flag), dec(base, flag)), (name, W, H, css, kw)
            n += 1
    assert n >= 40


def test_scripts_are_complete_and_valid():
    for ncomp in (3, 1):
        for name, script in PS.scripts(ncomp).items():
            al = np.full((ncomp, 64), -1)
            for comps, Ss, Se, Ah, Al in script:
                assert Ss <= Se and (Ss == 0) == (Se == 0) and (Ss == 0 or len(comps) == 1), name
                assert (al[list(comps), Ss:Se + 1] == (Ah if Ah else -1)).all(), (name, comps, Ss, Se, Ah)
                assert Ah == 0 or Al == Ah - 1
                al[list(comps), Ss:Se + 1] = Al
            assert (al == 0).all(), name
    assert len(PS.scripts(3)["per_coef"]) == 1 + 63 * 3
    assert max(s[4] for s in PS.scripts(3)["al10"]) == 10


def test_checkers_match_cv2_on_the_catalogue(oracle):
    for tag, jpg, ncomp in PS.catalogue(oracle, big=False):
        if ncomp == 3:
            assert np.array_equal(oracle.decode(jpg), dec(jpg)), tag
        assert np.array_equal(O.decode_gray(jpg), dec(jpg, cv2.IMREAD_GRAYSCALE)), tag


def test_incomplete_files_checkers(oracle):
    """a file libjpeg would smooth is refused (rc -18); every other one decodes to cv2's pixels"""
    n_refused = n_equal = 0
    for tag, jpg, ncomp, received in PS.incomplete(oracle):
        ref = with_eoi(jpg)
        for gray in ((False, True) if ncomp == 3 else (True,)):
            if PS.smoothed(received, ncomp, gray):
                with pytest.raises(RuntimeError, match="rc=-18"):
                    O.decode_gray(jpg) if gray else oracle.decode(jpg)
                n_refused += 1
            else:
                got = O.decode_gray(jpg) if gray else oracle.decode(jpg)
                assert np.array_equal(got, dec(ref, cv2.IMREAD_GRAYSCALE if gray else cv2.IMREAD_COLOR)), (tag, gray)
                n_equal += 1
    assert n_refused >= 100 and n_equal >= 60


def _pin_cases(oracle):
    """(tag, coef, qt, W, H, css, ncomp, script): complete scripts cut after every scan, and scripts that stop short"""
    comps = (0, 1, 2)
    short = {
        "only_10_63_unfinished": [(comps, 0, 0, 0, 0)] + [((c,), 1, 9, 0, 0) for c in comps] + [((c,), 10, 63, 0, 1) for c in comps],
        "only_dc_refinement_missing": [(comps, 0, 0, 0, 1)] + [((c,), 1, 63, 0, 0) for c in comps],
        "no_chroma_ac": [(comps, 0, 0, 0, 0), ((0,), 1, 63, 0, 0)],
        "no_cr_dc": [((0, 1), 0, 0, 0, 0)] + [((c,), 1, 63, 0, 1) for c in (0, 1)],
        "y_zz1_9_al1": [(comps, 0, 0, 0, 0)] + [((c,), 1, 63, 0, 0) for c in (1, 2)] + [((0,), 1, 9, 0, 1), ((0,), 10, 63, 0, 0)],
    }
    for name, script in short.items():
        coef, qt, W, H, _, _ = PS.entry(oracle, "simple", 57, 41, 3, seed=3, script=script)
        yield f"short/{name}", coef, qt, W, H, 3, 3, script
    for name, ncomp, W, H, css in (("simple", 3, 64, 48, 3), ("deep_sa", 3, 41, 29, 1), ("simple", 1, 40, 32, 0),
                                   ("dc_ycb_cr", 3, 48, 40, 0)):
        coef, qt, W, H, script, _ = PS.entry(oracle, name, W, H, css, ncomp, seed=4)
        for k in range(1, len(script) + 1):
            yield f"{name}/{ncomp}c/{W}x{H}/css{css}/{k} scans", coef, qt, W, H, css, ncomp, script[:k]


def test_smoothing_rule_pinned_to_cv2(oracle):
    """cv2 decodes a progressive file that stops after some scans exactly like a baseline file of the coefficients
    received so far whenever the rule says it does not smooth. Inside the rule smoothing runs, and it changes pixels
    unless every estimate it makes rounds to zero: most such files differ, on colour and on gray output."""
    h = J.std_huff(oracle)
    inside = {False: [], True: []}
    for tag, coef, qt, W, H, css, ncomp, script in _pin_cases(oracle):
        prog = PS.write_progressive(coef, qt, W, H, css, script, ncomp=ncomp, oracle=oracle)
        lay = PS.Layout(W, H, css, ncomp, oracle)
        base = J.write_baseline(PS.partial_coefs(coef, script, ncomp, lay=lay), qt, W, H, css, ncomp=ncomp, htabs=h, oracle=oracle)
        for gray in ((False, True) if ncomp == 3 else (True,)):
            flag = cv2.IMREAD_GRAYSCALE if gray else cv2.IMREAD_COLOR
            same = np.array_equal(dec(prog, flag), dec(base, flag))
            if PS.smoothed(script, ncomp, gray):
                inside[gray].append(not same)
            else:
                assert same, (tag, "gray" if gray else "colour")
    for gray, d in inside.items():
        assert len(d) >= 10 and sum(d) >= 0.75 * len(d), (gray, sum(d), len(d))
