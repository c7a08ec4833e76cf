#!/usr/bin/env python3
"""Regenerates tests/golden/streams.json by running the UNMODIFIED reference (oracle/_ref/libdsv1ref.so,
built by oracle/Makefile from the reference's source tree, its REF) on SURVEY.md Appendix-C synthetic content.

output_options.json pins the decoder's output options (debug overlay, 4:2:0 conversion) the same way.

Each entry pins: md5 of the input yuv, md5 + length of the reference .dsv stream (CRF, -rc_mode1 in CLI
terms) and md5 of the reference decoder's output.  Run:  python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import dsvlibs as L  # noqa: E402

CASES = [
    # name, w, h, fmt, frames, seed, cut, gop, qp
    ("cif_gop12", 352, 288, "420", 300, 1, 150, 12, 85),
    ("cif_gop0_24", 352, 288, "420", 24, 1, 0, 0, 85),
    ("qcif_gop12_444", 176, 144, "444", 30, 4, 14, 12, 85),
    ("qcif_gop12_422", 176, 144, "422", 26, 5, 0, 12, 70),
    ("qcif_gop12_411", 176, 144, "411", 26, 6, 0, 12, 95),
    ("w428_gop12", 428, 240, "420", 14, 7, 0, 12, 85),
    ("w854_gop6", 854, 480, "420", 8, 8, 0, 6, 85),
    ("hd_gop0", 1920, 1080, "420", 24, 2, 0, 0, 85),
    ("hd_gop12", 1920, 1080, "420", 24, 2, 0, 12, 85),
    ("hd_gop12_qp50", 1920, 1080, "420", 13, 9, 6, 12, 50),
    ("uhd444_gop12", 3840, 2160, "444", 6, 3, 0, 12, 85),
]


# decoder output options (CLI -drawinfo / -out420p): name, w, h, fmt, frames, seed, cut, gop, qp, extra cfg
OUTPUT_CASES = [
    ("cif_overlay", 352, 288, "420", 8, 21, 4, 12, 30, {}),
    ("edge_intra_444", 200, 120, "444", 4, 5, 2, 12, 60, dict(do_scd=0, intra_pct=100)),  # intra dots spill past luma
    ("edge_intra_422", 208, 104, "422", 4, 7, 2, 12, 40, dict(do_scd=0, intra_pct=100)),
    ("qcif_411", 176, 144, "411", 5, 6, 0, 12, 95, {}),
    ("hd_444", 1920, 1080, "444", 4, 9, 2, 12, 70, dict(do_scd=0, intra_pct=100)),
]


def output_options(ref):
    out = {}
    for name, w, h, fmt, n, seed, cut, gop, qp, kw in OUTPUT_CASES:
        yuv = L.synth_sequence(w, h, fmt, n, seed, cut)
        cfg = L.make_cfg(w, h, fmt, gop=gop, qp=qp, **kw)
        stream, _, _ = ref.encode_sequence(cfg, yuv, n)
        e = dict(w=w, h=h, fmt=fmt, frames=n, seed=seed, cut=cut, gop=gop, qp=qp, cfg=kw,
                 dsv_md5=hashlib.md5(stream).hexdigest(), dec={})
        for draw in (0, 1, 2, 4, 7):
            for to420 in (0, 1):
                nf, dec, _, _ = ref.decode_stream(stream, w, h, L.SUBSAMP[fmt], n, draw_info=draw, to_420p=to420)
                assert nf == n
                e["dec"]["draw%d_420p%d" % (draw, to420)] = hashlib.md5(dec.tobytes()).hexdigest()
        out[name] = e
        print(name, e["dsv_md5"], flush=True)
    json.dump(out, open(os.path.join(HERE, "output_options.json"), "w"), indent=1, sort_keys=True)


def main():
    ref = L.ref()
    if "--outputs-only" in sys.argv:
        output_options(ref)
        return
    output_options(ref)
    out = {}
    for name, w, h, fmt, n, seed, cut, gop, qp in CASES:
        yuv = L.synth_sequence(w, h, fmt, n, seed, cut)
        cfg = L.make_cfg(w, h, fmt, gop=gop, qp=qp)
        stream, pk, _ = ref.encode_sequence(cfg, yuv, n)
        nf, dec, meta, _ = ref.decode_stream(stream, w, h, L.SUBSAMP[fmt], n)
        assert nf == n
        out[name] = dict(w=w, h=h, fmt=fmt, frames=n, seed=seed, cut=cut, gop=gop, qp=qp,
                         yuv_md5=hashlib.md5(yuv.tobytes()).hexdigest(),
                         dsv_md5=hashlib.md5(stream).hexdigest(), dsv_len=len(stream), packets=len(pk),
                         dec_md5=hashlib.md5(dec.tobytes()).hexdigest())
        print(name, out[name]["dsv_md5"], len(stream), flush=True)
    json.dump(out, open(os.path.join(HERE, "streams.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
