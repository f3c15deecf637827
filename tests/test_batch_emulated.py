"""CPU tests of the BATCHED kernel sources (prepare_depth_batch_kernel, render_ao_batch_kernel, blur_upsample[_premin]_batch_kernel:
meao_render_batch) through the host emulator (tests/emu, with the 3-D TMA of tests/emu_batch), bit for bit against the oracle frame by frame.  B = 3 distinct frames at
ragged sizes, so every frame has border tiles and the tile index of the upsample crosses frame boundaries; the emulated 3-D tensor
map zero-fills per frame like cp.async.bulk.tensor.3d."""
import numpy as np
import pytest

from miniengineao_b200 import synth
from oracle.oracle import Oracle

from emu_batch.emu_batch import EmulatedBatch  # noqa: E402  (tests/ is on sys.path via conftest)
from test_kernel_logic_emulated import _plan  # noqa: E402


def _frames(W, H, B=3, seed=1):
    out = []
    for f in range(B):
        d = synth.lin01_to_raw(synth.random_depth(W, H, seed=seed + 37 * f))
        if W > 16 and H > 16 and f == 1:
            d[H // 4:H // 2, W // 4:W // 2] = 0.0         # sky in the middle frame: the IEEE fallbacks
        out.append(d)
    return np.stack(out)


def _check(f, depth, got, tag, ids=tuple(range(1, 17)), single_scale=False, **okw):
    orc = Oracle(depth.shape[2], depth.shape[1], threads=4, single_scale=single_scale, **okw)
    for fr in range(depth.shape[0]):
        ref = orc.run(depth[fr])
        assert np.array_equal(got[fr], ref), (tag, fr)
        for bid in ids:
            g = f.batch_buffer(fr, bid)
            if g.dtype == np.uint8:
                want = orc.codes(bid)
                assert np.array_equal(g, want), (tag, fr, bid)
            elif g.dtype == np.float16:
                with np.errstate(over="ignore"):
                    assert np.array_equal(g.view(np.uint16), orc.buffer(bid).astype(np.float16).view(np.uint16)), (tag, fr, bid)
            else:
                assert np.array_equal(g.view(np.uint32), orc.buffer(bid).view(np.uint32)), (tag, fr, bid)


@pytest.mark.parametrize("use_tma", [True, False])
@pytest.mark.parametrize("W,H", [(3, 5), (83, 61), (130, 70)])
def test_batch_reference_path(W, H, use_tma):
    d = _frames(W, H, seed=W + H)
    f = EmulatedBatch(_plan(W, H, intensity=1.1), use_tma=use_tma)
    _check(f, d, f.run_batch(d), f"{W}x{H} tma={use_tma}", intensity=1.1)


@pytest.mark.parametrize("use_tma", [True, False])
def test_batch_interior_tiles_and_forced_tile_loop(use_tma, monkeypatch):
    """Large enough for TMA-fed (interior) tiles in every frame; the persistent tile loop forced on every level, so one CTA walks
    the tiles of all three frames and prefetches across frame boundaries.  HQ mask 15 + exhaustive: the wide render and premin boxes."""
    monkeypatch.setenv("MEAO_UPS_PERSIST_MIN_WAVES", "0.0001")
    W, H = 640, 360
    d = _frames(W, H, seed=5)
    f = EmulatedBatch(_plan(W, H, intensity=1.2, high_quality_mask=15, sample_exhaustively=True), use_tma=use_tma)
    n0 = f.tma_box_loads()
    got = f.run_batch(d)
    assert (f.tma_box_loads() - n0 > 300) if use_tma else (f.tma_box_loads() == n0)
    _check(f, d, got, f"variants tma={use_tma}", tuple(range(1, 17)) + (18, 19, 20, 21),
           intensity=1.2, high_quality_mask=15, sample_exhaustively=True)


@pytest.mark.parametrize("W,H", [(130, 70), (83, 61)])
def test_batch_single_scale(W, H):
    d = _frames(W, H, seed=9)
    plan = _plan(W, H, intensity=1.1)
    plan.singleScale = True
    f = EmulatedBatch(plan)
    _check(f, d, f.run_batch(d), "single_scale", ids=(1, 2, 3, 4, 5, 10), single_scale=True, intensity=1.1)


def test_plan_only_context_refuses_render_batch():
    import ctypes as C
    from miniengineao_b200 import AmbientOcclusion, Camera
    from miniengineao_b200 import _native as N
    p = AmbientOcclusion(Camera(64, 32), device=-1)
    p.LateUpdate()
    buf = (C.c_float * (2 * 64 * 32))()
    out = (C.c_uint8 * (2 * 64 * 32))()
    assert N.lib().meao_render_batch(p._ctx, buf, N.MEAO_DEPTH_RAW_F32, 2, out, None) == N.MEAO_ERR_CUDA
    assert N.lib().meao_reserve_batch(p._ctx, 2) == N.MEAO_ERR_CUDA
