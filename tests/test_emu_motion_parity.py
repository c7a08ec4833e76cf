"""The motion kernels configured as EncEngine::step / DecEngine::step launch them (ingest with border, batched pyramid,
luma sum, search over several lanes, out-of-place compensation from the reconstruction, the code pass, the decoder's
in-place compensation of the P lanes), on the test-only CPU emulation of the same sources, against the plain-C port.
Small sizes; the device runs them at full size in test_gpu_motion_parity.py."""
import subprocess

import pytest

import dsvlibs as L
import motionparity as MP

# w % 16 in {0, 2, 6, 8, 14}; odd chroma widths and chroma widths that are no multiple of 16; odd pyramid levels;
# the codec's block sizes and the BMC strip cases' explicit ones.  (No 4:1:1 picture whose last block column is 2
# samples wide: its chroma is 0 samples wide there, and the port, like the reference, divides by zero in the search.)
GEOMS = [  # w, h, format, block size (None: the codec's), lanes (the emulator's time goes with lanes x calls)
    (16, 16, "420", None, 2),
    (50, 34, "420", None, 4),        # w % 16 = 2, chroma 25 x 17
    (52, 34, "411", None, 1),        # chroma 13 wide, its edge block 1 wide
    (54, 38, "420", None, 2),        # w % 16 = 6, chroma 27 x 19, levels 27 / 14 / 7
    (62, 34, "420", None, 1),        # w % 16 = 14, chroma 31 wide: one byte of stride tail per row
    (60, 32, "411", None, 1),        # chroma 15 wide
    (72, 40, "422", (24, 16), 3),    # w % 16 = 8, chroma 36 wide
    (78, 46, "444", (20, 28), 1),    # w % 16 = 14
    (132, 52, "420", (64, 48), 1),
    (108, 70, "411", (36, 20), 2),   # chroma 27 wide
    (200, 120, "422", None, 1),      # w % 16 = 8, chroma 100 wide
]
ids = lambda g: f"{g[0]}x{g[1]}_{g[2]}_{'auto' if g[3] is None else '%dx%d' % g[3]}_n{g[4]}"  # noqa: E731

# (has_ref, do_sum) per lane and call: every lane starts without a reference; later calls mix I lanes (before P lanes
# too), P lanes with and without a sum, sums without a search
SCHEDULES = {
    1: [[(0, 1)], [(1, 1)], [(1, 0)]],
    2: [[(0, 0), (0, 1)], [(0, 1), (1, 1)], [(1, 0), (1, 1)]],
    3: [[(0, 1), (0, 0), (0, 1)], [(1, 1), (0, 0), (1, 0)], [(0, 1), (1, 1), (1, 1)]],
    4: [[(0, 1), (0, 1), (0, 0), (0, 1)], [(0, 1), (1, 1), (1, 0), (1, 1)], [(1, 1), (0, 0), (1, 1), (1, 0)]],
}


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", L.PKG, "emu"], check=True, stdout=subprocess.DEVNULL)
    return L.emu()


@pytest.mark.parametrize("geom", GEOMS, ids=ids)
def test_motion_lanes_emu(emu, port, geom):
    w, h, fmt, blk, n = geom
    kinds = ["synth"] * n
    if n > 2:
        kinds[1] = "noise"  # unlike its neighbours: a lane mix-up changes every output
    MP.run_sequence(emu, port, MP.Geom(w, h, fmt, blk), SCHEDULES[n], seed=w + h, kinds=kinds, device_src=MP.at_offset)


def test_motion_scene_cut_emu(emu, port):
    """two lanes of different content at a size whose pyramid has odd levels in both directions; lane 0 cuts to a new
    scene at its third picture (most blocks intra there)"""
    g = MP.Geom(70, 46, "420")
    cuts = [2, 0]
    MP.run_sequence(emu, port, g, SCHEDULES[2], seed=5, device_src=MP.at_offset,
                    content_fn=lambda k, t: L.synth_sequence(g.w, g.h, g.fmt, 1, 5 + k, cuts[k], start=t))


def test_motion_reject_emu(emu):
    MP.check_reject(emu, MP.Geom(54, 38, "420"))


@pytest.mark.parametrize("geom", GEOMS, ids=ids)
def test_decoder_compensation_emu(emu, port, geom):
    w, h, fmt, blk, _ = geom
    MP.run_decoder(emu, port, MP.Geom(w, h, fmt, blk), isP=[0, 1, 1, 0, 1], seed=w * h)
