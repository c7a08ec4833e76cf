"""oracle/dsv1_port.c subband transform == unmodified reference (sbt.c), exact integers."""
import numpy as np
import pytest

import refdigest

SIZES = [  # (plane w, plane h, coef w, coef h)
    (60, 34, 60, 34), (120, 68, 120, 68), (54, 86, 54, 86), (352, 288, 352, 288), (176, 144, 176, 144),
    (427, 240, 428, 240), (959, 539, 960, 540), (135, 67, 136, 68), (16, 16, 16, 16), (480, 270, 480, 270),
]


def content(rng, ph, cols, kind):
    if kind == "noise":
        return rng.integers(0, 256, size=(ph, cols), dtype=np.uint8)
    y, x = np.mgrid[0:ph, 0:cols]
    v = 128 + 60 * np.sin(x / 9.0) + 50 * np.cos(y / 7.0) + rng.integers(-6, 7, size=(ph, cols))
    return np.clip(v, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("dims", SIZES)
@pytest.mark.parametrize("isP", [0, 1])
def test_fwd_inv(ref, port, dims, isP):
    pw, ph, cw, ch = dims
    rng = np.random.default_rng(pw * 31 + ph + isP)
    for kind in ("noise", "smooth"):
        pix = content(rng, ph, cw + 2, kind)
        a = ref.fwd_sbt(pix, pw, ph, cw, ch, isP)
        b = port.fwd_sbt(pix, pw, ph, cw, ch, isP)
        assert np.array_equal(a, b)
        for step in (1, 9, 40):
            co = (a // step) * step
            for c in (0, 1):
                for q in (313, 1200):
                    assert np.array_equal(ref.inv_sbt(co, q, isP, c, pw, ph), port.inv_sbt(co, q, isP, c, pw, ph))


def test_hd_luma(ref, port):
    rng = np.random.default_rng(7)
    pix = content(rng, 1080, 1920, "smooth")
    for isP in (0, 1):
        a = ref.fwd_sbt(pix, 1920, 1080, 1920, 1080, isP)
        assert np.array_equal(a, port.fwd_sbt(pix, 1920, 1080, 1920, 1080, isP))
        co = (a // 16) * 16
        assert np.array_equal(ref.inv_sbt(co, 313, isP, 0, 1920, 1080), port.inv_sbt(co, 313, isP, 0, 1920, 1080))


def _quant_tables(lib):
    quant = [lib.fn("get_quant")(q, isP, lvl) for q in range(0, 2048, 7) for isP in (0, 1) for lvl in (0, 1, 2)]
    lb2 = [lib.fn("lb2")(n) for n in list(range(0, 70)) + [255, 256, 257, 4095, 4096, 4097, 1 << 20]]
    return quant, lb2


def test_quant_tables(ref, port):
    assert refdigest.table(ref, "quant_tables", _quant_tables) == _quant_tables(port)
