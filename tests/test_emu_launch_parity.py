"""The transform and entropy-coding kernels configured as EncEngine::step / DecEngine::step launch them (tile flags, list
scratch, fused prediction add, multi-picture mapping, carried decoder state), on the test-only CPU emulation of the same
sources, against the plain-C port.  Small sizes; the same cases at full size run on the device in
test_gpu_launch_parity.py."""
import subprocess

import numpy as np
import pytest

import dsvlibs as L
import launchparity as LP

GEOMS = [(16, 16, "420"), (54, 38, "420"), (136, 68, "444"), (214, 120, "422"), (384, 192, "420"), (428, 240, "411"),
         (520, 200, "420")]


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


def run_encode_parity(lib, port, w, h, fmt, npics, seed, calls=2, check=None):
    """check: the pictures compared with the port (default all of them)"""
    g = LP.Geom(w, h, fmt)
    enc = LP.Enc(lib, g, npics)
    try:
        starts = [0, 1, 3, 13, 4093]
        # call 1: long pictures (fine quantiser), call 2 on the same lanes: short ones (coarse), so that the second call
        # relies on the dirty-prefix clean-up of the first call's packets, list scratch and flags
        for call, qps in enumerate(((100, 85), (50, 85))[:calls]):
            pics, ins, preds = LP.content(g, npics, seed + call, qps=qps)
            for k, p in enumerate(pics):
                p["start_byte"] = starts[(k + call) % len(starts)]
                p["cap"] = enc.pkt_bytes
            out = enc.run(pics, ins, preds)
            LP.check_encode(port, enc, pics, ins, preds, out, check)
            if call == 0:
                first_total = out["info"][:, 1].copy()
        if calls > 1:
            assert (out["info"][:, 1] < first_total).any(), "the second call should be shorter in some lane"
    finally:
        enc.close()


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: f"{g[0]}x{g[1]}_{g[2]}")
def test_encode_parity_emu(emu, port, geom):
    # the two-call sequence on the five smaller formats; the device runs it on every format
    run_encode_parity(emu, port, *geom, npics=3, seed=geom[0], calls=1 if geom[0] * geom[1] > 384 * 192 else 2)


def run_overflow(lib, port, w, h, fmt, npics, seed):
    """One picture of a call gets a cap just below its coded size: it reports overflow and writes nothing at or past the
    cap; the others stay byte-exact."""
    g = LP.Geom(w, h, fmt)
    enc = LP.Enc(lib, g, npics)
    try:
        pics, ins, preds = LP.content(g, npics, seed, qps=(100,))
        for p in pics:
            p["start_byte"], p["cap"] = 13, enc.pkt_bytes
        sizes = enc.run(pics, ins, preds)["info"][:, 1]
        victim = npics // 2
        pics[victim]["cap"] = int(sizes[victim]) - 1
        out = enc.run(pics, ins, preds)
        assert out["info"][victim, 0] == 1, "a picture one byte over its cap must report overflow"
        assert not out["pkt"][victim, pics[victim]["cap"]:].any(), "bytes written at or past the cap"
        LP.check_encode(port, enc, pics, ins, preds, out, check=set(range(npics)) - {victim})
        pics[victim]["cap"] = enc.pkt_bytes  # the lane recovers on the next call
        LP.check_encode(port, enc, pics, ins, preds, enc.run(pics, ins, preds))
    finally:
        enc.close()


def test_overflow_emu(emu, port):
    run_overflow(emu, port, 214, 120, "422", 3, 11)


def run_list_edges(lib, port, seed):
    """HZCC chunks at the edges of the list scratch, I (sparse and dense lists) and P (sparse lists) in one launch:
    127 / 128 / 129 marked groups with one non-zero each and with four (127 x 4 = 508 fills a sparse list exactly),
    non-zeros on both sides of a chunk boundary, chunks of bands whose tiles are flagged empty beside flagged ones,
    all-zero chroma planes.  Then a negative control: a flag cleared over a non-zero must change the stream."""
    g = LP.Geom(384, 192, "420")
    rng = np.random.default_rng(seed)
    pics, raws, flags, exp = [], [], [], []
    for isP in (0, 1):
        pic = dict(isP=isP, quant=LP.quant_of_qp(100), stable=np.zeros(g.nbh * g.nbv, np.uint8), start_byte=7 + 6 * isP)
        planes = LP.list_edge_planes(g, rng)
        res = [port.encode_plane(co, pic["quant"], isP, c, pic["stable"], g.nbh, g.nbv) for c, co in enumerate(planes)]
        y = res[0][1]
        for chunk, (groups, per) in LP.LIST_EDGE_CHUNKS.items():
            assert LP.marked_groups(y, chunk) == (groups, groups * per), (chunk, LP.marked_groups(y, chunk))
        xs, ys = LP.scan_map(384, 192)
        assert all(y[ys[p_], xs[p_]] for p_ in LP.BOUNDARY_POSITIONS)
        fl = [LP.exact_flags(d) for _, d in res]
        assert not (fl[0][2] & 1).any() and not (fl[0] & 2).any() and not fl[1].any() and not fl[2].any()
        pics.append(pic)
        raws.append(planes)
        flags.append(fl)
        exp.append(res)
    cap = LP.Enc(lib, g, 1)
    for p in pics:
        p["cap"] = cap.pkt_bytes
    cap.close()
    pkt, info, deq, dv = LP.hz_enc_batch(lib, g, pics, raws, flags)
    for k, pic in enumerate(pics):
        body = np.concatenate([b for b, _ in exp[k]])
        sb = pic["start_byte"]
        assert info[k, 0] == 0 and info[k, 1] == sb + len(body), (k, info[k])
        assert np.array_equal(pkt[k, sb:info[k, 1]], body), f"picture {k} (isP={pic['isP']}): stream differs from the port"
        assert not pkt[k, :sb].any() and not pkt[k, info[k, 1]:].any(), f"picture {k}: bytes outside the packet"
        for c, d in enumerate(g.split_coef(deq[k])):
            assert np.array_equal(d, exp[k][c][1]), (k, c)
    # negative control: level-1 flags of luma tile row 0 cleared over the non-zeros of chunk 9 -> the chunk is skipped
    cleared = [[f.copy() for f in fl] for fl in flags]
    for fl in cleared:
        fl[0][0] &= 0xFE
    pkt2, info2, _, _ = LP.hz_enc_batch(lib, g, pics[:1], raws[:1], cleared[:1])
    for k in range(1):
        assert not np.array_equal(pkt2[k, :info2[k, 1]], pkt[k, :info[k, 1]]), \
            f"picture {k}: a cleared level-1 flag over non-zeros did not change the stream (the skip is not taken)"


def test_hzcc_list_edges_emu(emu, port):
    run_list_edges(emu, port, 3)


def test_double_visited_first_visits_emu(emu, port):
    """Luma 454 wide: level-1 bands 227 wide, so the level-2 scan also visits the first column of LH1 / HH1 and takes
    those first visits from the side buffer.  The residual has a step between pixel columns 0 and 1 only: level 2 is
    empty (its tiles flagged so) while that column is not, and every chunk inside the level-2 bands must still be coded."""
    g = LP.Geom(454, 256, "420")
    enc = LP.Enc(emu, g, 1)
    try:
        res = np.full(g.frame_bytes, 128, dtype=np.uint8)
        y = res[:454 * 256].reshape(256, 454)
        y[:, 0], y[:, 1] = 128 + 60, 128 - 60
        pic = dict(isP=1, quant=LP.quant_of_qp(100), stable=np.zeros(g.nbh * g.nbv, np.uint8), start_byte=5, cap=enc.pkt_bytes)
        out = enc.run([pic], [res], [np.full(g.frame_bytes, 100, np.uint8)])
        co = g.split_coef(out["coef"][0])[0]
        assert co[:, 227].any() and not (LP.exact_flags(co) & 2).any()
        LP.check_encode(port, enc, [pic], [res], [np.full(g.frame_bytes, 100, np.uint8)], out)
    finally:
        enc.close()


def hand_planes(g, rng):
    """Sparse coefficient planes with non-zeros where the flag mechanism can go wrong: tile corners, a neighbour's level-2
    blocks only, the last partial tile column / row, the double-visited edge positions."""
    out = []
    for cw, ch in g.coefs:
        co = np.zeros((ch, cw), dtype=np.int32)
        co[0, 0] = 700
        co[:2, :2] += rng.integers(-300, 300, size=(2, 2), dtype=np.int32)
        wo1, ho1 = cw // 2, ch // 2
        wo2, ho2 = -(-wo1 // 2), -(-ho1 // 2)
        # level 1: every corner of the first and of the last (partial) tile's blocks in HH1 / LH1 / HL1
        for (x0, y0, bw, bh) in ((wo1, ho1, cw - wo1, ch - ho1), (wo1, 0, cw - wo1, ho1), (0, ho1, wo1, ch - ho1)):
            for bx in (0, 63, bw - 1):
                for by in (0, 31, bh - 1):
                    if bx < bw and by < bh:
                        co[y0 + by, x0 + bx] = int(rng.choice([-1, 1])) * int(rng.integers(40, 900))
        # level 2: only the block of tile (1, 0) / (0, 1) -- its neighbours rely on the halo union of the flags
        for (x0, y0, bw, bh) in ((wo2, ho2, wo1 - wo2, ho1 - ho2), (wo2, 0, wo1 - wo2, ho2), (0, ho2, wo2, ho1 - ho2)):
            for bx, by in ((32, 0), (0, 16), (31, 15), (bw - 1, bh - 1)):
                if bx < bw and by < bh:
                    co[y0 + by, x0 + bx] = int(rng.integers(-500, 500)) or 9
        # double-visited positions: the column / row just past an odd level-2 band
        if wo2 & 1 or ho2 & 1:
            co[min(ho1 - 1, ho2), min(wo1 - 1, wo2)] = 333
        out.append(co)
    return out


def run_inverse_flags(lib, port, w, h, fmt, seed):
    g = LP.Geom(w, h, fmt)
    rng = np.random.default_rng(seed)
    seq = LP.frame_content(g, seed, 0, rng)
    geoms, pics, coefs, flags, preds, variants = [], [], [], [], [], []
    for isP in (0, 1):
        for variant in ("exact", "all", "superset"):
            planes = hand_planes(g, rng)
            ex = [LP.exact_flags(c) for c in planes]
            if variant == "all":
                fl = [np.full_like(e, 3) for e in ex]
            elif variant == "superset":
                fl = [e | rng.integers(0, 4, size=e.shape, dtype=np.uint8) for e in ex]
            else:
                fl = ex
            geoms.append(g)
            pics.append(dict(isP=isP, quant=LP.quant_of_qp((85, 50, 100)[len(pics) % 3])))
            coefs.append(np.concatenate([c.ravel() for c in planes]))
            flags.append(np.concatenate([f.ravel() for f in fl]))
            preds.append(seq)
            variants.append(variant)
    for with_pred in (False, True):
        got = LP.inv_batch(lib, geoms, pics, coefs, flags, preds if with_pred else None)
        for k, pic in enumerate(pics):
            for c, (co, rec) in enumerate(zip(g.split_coef(coefs[k]), g.split_frame(got[k]))):
                pw, ph = g.planes[c]
                pr = g.split_frame(seq)[c] if with_pred and pic["isP"] else None  # the engines add it to P pictures only
                want = LP.recon_ref(port, co, pic["quant"], pic["isP"], c, pw, ph, pr)
                assert np.array_equal(rec, want), (k, c, variants[k], pic, with_pred)
    return g, geoms, pics, coefs, flags


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: f"{g[0]}x{g[1]}_{g[2]}")
def test_inverse_with_flags_emu(emu, port, geom):
    run_inverse_flags(emu, port, *geom, seed=geom[1])


def run_negative_inverse(lib, port, w, h, fmt, isP):
    """A cleared flag over a tile that holds a non-zero must change the output: the skip path is really taken."""
    g = LP.Geom(w, h, fmt)
    cw, ch = g.coefs[0]
    planes = [np.zeros((c[1], c[0]), dtype=np.int32) for c in g.coefs]
    # level 1, HH band, interior tile (1, 1) where the plane has one
    tx, ty = (1, 1) if cw >= 384 and ch >= 192 else (0, 0)
    planes[0][ch // 2 + ty * 32 + 5, cw // 2 + tx * 64 + 7] = 2000
    fl = [LP.exact_flags(c) for c in planes]
    assert fl[0][ty, tx] & 1
    cleared = [f.copy() for f in fl]
    cleared[0][ty, tx] &= 0xFE
    pic = dict(isP=isP, quant=LP.quant_of_qp(100))
    co = np.concatenate([c.ravel() for c in planes])
    good, bad = LP.inv_batch(lib, [g, g], [pic, pic], [co, co],
                             [np.concatenate([f.ravel() for f in fl]), np.concatenate([f.ravel() for f in cleared])])
    want = LP.recon_ref(port, planes[0], pic["quant"], isP, 0, w, h)
    assert np.array_equal(g.split_frame(good)[0], want)
    assert not np.array_equal(g.split_frame(bad)[0], want), "a cleared level-1 flag did not change the output"


def test_negative_control_inverse_emu(emu, port):
    # P picture: the compile-time-geometry path of an interior tile (I pictures read level 1 whatever the flags say)
    run_negative_inverse(emu, port, 384, 192, "420", 1)


def run_decoder_state(lib, port, w, h, fmt, seed):
    """One decoder lane over I (dense), P, P (level-1 content in other tiles), I, P with a truncated plane, P."""
    g = LP.Geom(w, h, fmt)
    rng = np.random.default_rng(seed)
    dec = LP.Dec(lib, g)
    q_i, q_p = LP.quant_of_qp(50), LP.quant_of_qp(100)
    try:
        for k, kind in enumerate(("I", "P", "P2", "I", "Ptrunc", "P")):
            isP = kind != "I"
            stable = rng.integers(0, 4, size=g.nbh * g.nbv, dtype=np.uint8)
            pic = dict(isP=int(isP), quant=q_p if isP else q_i, stable=stable)
            recs, ref_coefs = [], []
            for c, (cw, ch) in enumerate(g.coefs):
                if kind == "I":  # every position drawn; the second I picture sparser, so that tiles empty out
                    co = (rng.laplace(0, 300, size=(ch, cw)) * (rng.random((ch, cw)) < (1.0 if k == 0 else 0.3))).astype(np.int32)
                else:
                    co = np.zeros((ch, cw), dtype=np.int32)
                    dens = rng.random((ch, cw)) < 0.01
                    co[dens] = rng.integers(-3000, 3000, size=int(dens.sum()))
                    # level-1 content in a varying subset of tiles, so that tiles go from non-zero to empty
                    ty_, tx_ = -(-ch // 64), -(-cw // 128)
                    keep = rng.random((ty_, tx_)) < (0.5 if kind == "P2" else 0.2)
                    m = np.zeros((ch, cw), dtype=bool)
                    for yy in range(ty_):
                        for xx in range(tx_):
                            if not keep[yy, xx]:
                                m[ch // 2 + yy * 32: ch // 2 + yy * 32 + 32, cw // 2 + xx * 64: cw // 2 + xx * 64 + 64] = True
                                m[ch // 2 + yy * 32: ch // 2 + yy * 32 + 32, xx * 64: min(cw // 2, xx * 64 + 64)] = True
                                m[yy * 32: min(ch // 2, yy * 32 + 32), cw // 2 + xx * 64: cw // 2 + xx * 64 + 64] = True
                    co[m] = 0
                    co[0, 0] = int(rng.integers(-2000, 2000))
                data, _ = port.encode_plane(co, pic["quant"], pic["isP"], c, stable, g.nbh, g.nbv)
                data = bytearray(data.tobytes())
                if kind == "Ptrunc" and c == 2:
                    plen = int.from_bytes(data[:4], "big")
                    cut = max(plen // 3, min(plen, 16))  # past the plane head: a cut DC is not this test's subject
                    data = bytearray(cut.to_bytes(4, "big")) + data[4:4 + cut]
                recs.append(bytes(data))
                ref_coefs.append(port.decode_plane(np.frombuffer(bytes(data), np.uint8), cw, ch, pic["quant"], pic["isP"], c,
                                                   stable, g.nbh, g.nbv))
            n, coef, tfl = dec.run(pic, b"".join(recs))
            assert n == 3
            for c, (got, want, fl) in enumerate(zip(g.split_coef(coef), ref_coefs, g.split_flags(tfl))):
                assert np.array_equal(got, want), f"picture {k} ({kind}) plane {c}: decoded coefficients"
                LP.check_dec_flags(fl, got, f"picture {k} ({kind}) plane {c}")
    finally:
        dec.close()


@pytest.mark.parametrize("geom", GEOMS, ids=lambda g: f"{g[0]}x{g[1]}_{g[2]}")
def test_decoder_carried_state_emu(emu, port, geom):
    run_decoder_state(emu, port, *geom, seed=geom[0] + geom[1])
