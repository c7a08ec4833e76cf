"""The transform and entropy-coding kernels configured as EncEngine::step / DecEngine::step launch them, on the B200,
against the plain-C port: the cases of test_emu_launch_parity.py at full size, plus the bench's launch shape (64 HD
pictures in one call: 192 jobs with the arithmetic tile mapping and HzMap) and a call whose pictures differ in tile
count (binary-search mapping)."""
import numpy as np
import pytest

import launchparity as LP
from test_emu_launch_parity import GEOMS, run_decoder_state, run_encode_parity, run_inverse_flags, run_list_edges, run_negative_inverse, run_overflow

GPU_GEOMS = GEOMS + [(1280, 720, "422"), (854, 480, "411")]
ids = lambda g: f"{g[0]}x{g[1]}_{g[2]}"  # noqa: E731


@pytest.mark.gpu
@pytest.mark.parametrize("geom", GPU_GEOMS, ids=ids)
def test_encode_parity_gpu(gpu, port, geom):
    run_encode_parity(gpu, port, *geom, npics=4, seed=geom[0])


@pytest.mark.gpu
def test_encode_parity_bench_shape_gpu(gpu, port):
    # one call of 64 pictures; the port (a CPU coder) checks an I/P pair out of every 8 lanes, first and last included
    run_encode_parity(gpu, port, 1920, 1080, "420", npics=64, seed=7, calls=1, check={k for k in range(64) if k % 8 < 2 or k >= 62})


@pytest.mark.gpu
def test_encode_parity_uhd_444_gpu(gpu, port):
    run_encode_parity(gpu, port, 3840, 2160, "444", npics=4, seed=9, calls=1)


@pytest.mark.gpu
@pytest.mark.parametrize("geom", GPU_GEOMS, ids=ids)
def test_inverse_with_flags_gpu(gpu, port, geom):
    run_inverse_flags(gpu, port, *geom, seed=geom[1])


@pytest.mark.gpu
def test_inverse_mixed_formats_gpu(gpu, port):
    """Pictures of different formats in one launch: the tile -> job mapping falls back to the binary search."""
    rng = np.random.default_rng(5)
    geoms = [LP.Geom(*g) for g in ((384, 192, "420"), (136, 68, "444"), (520, 200, "420"), (214, 120, "422"))]
    pics, coefs, flags = [], [], []
    for k, g in enumerate(geoms):
        planes = [(rng.laplace(0, 200, size=(ch, cw)) * (rng.random((ch, cw)) < 0.02)).astype(np.int32) for cw, ch in g.coefs]
        pics.append(dict(isP=k % 2, quant=LP.quant_of_qp(85)))
        coefs.append(np.concatenate([c.ravel() for c in planes]))
        flags.append(np.concatenate([LP.exact_flags(c).ravel() for c in planes]))
    got = LP.inv_batch(gpu, geoms, pics, coefs, flags)
    for k, (g, pic) in enumerate(zip(geoms, pics)):
        for c, (co, rec) in enumerate(zip(g.split_coef(coefs[k]), g.split_frame(got[k]))):
            pw, ph = g.planes[c]
            assert np.array_equal(rec, LP.recon_ref(port, co, pic["quant"], pic["isP"], c, pw, ph)), (k, c)


@pytest.mark.gpu
def test_hzcc_list_edges_gpu(gpu, port):
    run_list_edges(gpu, port, 3)


@pytest.mark.gpu
def test_overflow_gpu(gpu, port):
    run_overflow(gpu, port, 1280, 720, "422", 5, 11)


@pytest.mark.gpu
def test_negative_control_inverse_gpu(gpu, port):
    run_negative_inverse(gpu, port, 384, 192, "420", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("geom", GPU_GEOMS, ids=ids)
def test_decoder_carried_state_gpu(gpu, port, geom):
    run_decoder_state(gpu, port, *geom, seed=geom[0] + geom[1])
