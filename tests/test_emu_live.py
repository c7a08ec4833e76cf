"""Live streams (dsvb_enc_open / _push / _close, dsvb_dec_open / _push / _close, csrc/host/live.cpp) on the test-only
CPU emulation of the CUDA sources, at small sizes: streams pushed picture by picture through shared engine steps equal
the per-picture API's, ABR and intra-only objects included; the reports; every error path.  test_gpu_live.py runs
the golden vectors and device I/O on the B200."""
import subprocess

import pytest

import dsvlibs as L
import livelibs as LV


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


@pytest.mark.parametrize("gop", [3, 0])
def test_live_mixed_streams_emu(emu, gop):
    LV.check_mixed_streams(emu, 32, 32, "420", 2, [(4, 1, 0), (2, 2, 0), (4, 3, 2)], 10 + gop, gop=3 if gop else 0)


def test_live_abr_emu(emu):
    LV.check_mixed_streams(emu, 32, 32, "422", 2, [(4, 5, 2), (3, 6, 0), (3, 7, 0)], 20, gop=3, rc_mode=1,
                           bitrate=40000, quality=L.qp_to_quality(70) * 3 // 2)


def test_live_reports_emu(emu):
    LV.check_reports(emu, 32, 32, "444", 4, 3, 30, gop=3)


def test_live_encoder_errors_emu(emu):
    LV.check_encoder_errors(emu, 32, 32, "420")


def test_live_decoder_errors_emu(emu):
    LV.check_decoder_errors(emu, 32, 32, "420", 48, 32)
