"""GPU tests of batched rendering (AmbientOcclusion.render_batch / meao_render_batch): B independent frames in one call and one
graph replay.  Bar: bit-exact (TOL_CODES = 0) against the oracle on every frame's AO and on the intermediates of the first, a
middle and the last frame (batch_buffer), and equal to single-frame render() wherever the oracle would be slow."""
import numpy as np
import pytest

from test_parity_gpu import SIZES, _mk  # noqa: E402  (tests/ is on sys.path)

pytestmark = pytest.mark.gpu

TOL_CODES = 0


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a GPU")
    return torch


def _frames(W, H, B, seed, sky=False):
    from miniengineao_b200 import synth
    out = []
    for f in range(B):
        d = synth.lin01_to_raw(synth.random_depth(W, H, seed=seed + 101 * f))
        if sky and W > 8 and H > 8:
            d[H // 4:H // 2, W // 3:W // 2] = 0.0
        out.append(d)
    return np.stack(out)


def _compare_frame(ao, orc, f, ids, tag):
    bad = []
    for bid in ids:
        got = ao.batch_buffer(f, bid)
        ref = orc.buffer(bid)
        if got.dtype == np.uint8:
            n = int((np.abs(got.astype(np.int16) - orc.codes(bid).astype(np.int16)) > TOL_CODES).sum())
        elif got.dtype == np.float16:
            with np.errstate(over="ignore"):
                n = int((got.view(np.uint16) != ref.astype(np.float16).view(np.uint16)).sum())
        else:
            n = int((got.view(np.uint32) != ref.view(np.uint32)).sum())
        if n:
            bad.append((bid, n, got.size))
    assert not bad, f"{tag} frame {f}: mismatching buffers (id, #diff, size): {bad}"


def _check_batch(torch, ao, orc, depth_np, got, tag, ids=tuple(range(1, 17)), as_float=None):
    """Every frame's AO against the oracle; all `ids` of the first, a middle and the last frame."""
    B = depth_np.shape[0]
    inspect = sorted({0, B // 2, B - 1})
    for f in range(B):
        ref = orc.run(as_float[f] if as_float is not None else depth_np[f])
        assert int((np.abs(got[f].astype(np.int16) - ref.astype(np.int16)) > TOL_CODES).sum()) == 0, (tag, f)
        if f in inspect:
            _compare_frame(ao, orc, f, ids, tag)


@pytest.mark.parametrize("B", [1, 2, 5])
@pytest.mark.parametrize("W,H", SIZES)
def test_batch_sizes_bit_exact(torch_cuda, W, H, B):
    torch = torch_cuda
    ao, orc = _mk(W, H, intensity=1.1)
    d = _frames(W, H, B, seed=W * 7 + H)
    n0 = ao.launch_count
    got = ao.render_batch(torch.from_numpy(d).cuda()).cpu().numpy()
    assert got.shape == (B, H, W)
    assert ao.launch_count - n0 == ao.kernels_per_frame          # one frame's kernels per batch call
    _check_batch(torch, ao, orc, d, got, f"{W}x{H} B={B}")


VARIANTS = [
    dict(reversed_z=False),
    dict(single_pass_stereo=True),
    dict(sample_exhaustively=True),
    dict(high_quality_mask=8),
    dict(high_quality_mask=15, sample_exhaustively=True),
]


@pytest.mark.parametrize("variant", VARIANTS, ids=lambda v: "-".join(f"{k}={v[k]}" for k in v))
@pytest.mark.parametrize("W,H", [(322, 203), (1000, 37)])          # even widths: a stereo frame is an eye pair
def test_batch_variants_bit_exact(torch_cuda, W, H, variant):
    torch = torch_cuda
    ao, orc = _mk(W, H, intensity=1.1, **dict(variant))
    d = _frames(W, H, 3, seed=5, sky=True)
    if variant.get("reversed_z") is False:
        from miniengineao_b200 import synth
        d = np.stack([synth.lin01_to_raw(synth.random_depth(W, H, seed=5 + f), reversed_z=False) for f in range(3)])
    got = ao.render_batch(torch.from_numpy(d).cuda()).cpu().numpy()
    mask = variant.get("high_quality_mask", 0)
    ids = tuple(range(1, 17)) + tuple(17 + k for k in range(1, 5) if (mask >> (k - 1)) & 1)
    _check_batch(torch, ao, orc, d, got, str(variant), ids)


def test_batch_single_scale(torch_cuda):
    from miniengineao_b200 import AmbientOcclusion, Camera
    from oracle.oracle import Oracle
    torch = torch_cuda
    W, H = 330, 170
    d = _frames(W, H, 4, seed=3)
    ao = AmbientOcclusion(Camera(W, H), device=0)
    ao.intensity, ao.singleScale = 1.1, True
    got = ao.render_batch(torch.from_numpy(d).cuda()).cpu().numpy()
    orc = Oracle(W, H, threads=8, intensity=1.1, single_scale=True)
    _check_batch(torch, ao, orc, d, got, "single_scale", ids=(1, 2, 3, 4, 5, 10))


def test_batch_linear_and_native_depth_formats(torch_cuda):
    from miniengineao_b200 import synth
    torch = torch_cuda
    W, H = 250, 131
    lin = np.stack([synth.random_depth(W, H, seed=17 + f) for f in range(3)])
    ao, orc = _mk(W, H, intensity=1.1)
    got = ao.render_batch(torch.from_numpy(lin).cuda(), linear=True).cpu().numpy()
    from oracle.oracle import Oracle
    _check_batch(torch, ao, Oracle(W, H, threads=8, intensity=1.1, depth_is_linear=True), lin, got, "linear")
    raw = synth.lin01_to_raw(lin).astype(np.float64)
    for bits in (16, 24):
        ao, orc = _mk(W, H, intensity=1.1)
        full = (1 << bits) - 1
        codes = np.clip(np.rint(raw * full), 1, full).astype(np.uint32)
        as_float = (codes.astype(np.float32) * np.float32(1.0 / full)).astype(np.float32)
        if bits == 16:
            dev = torch.from_numpy(codes.astype(np.uint16).view(np.int16)).cuda().view(torch.uint16)
        else:
            dev = torch.from_numpy((codes | (np.uint32(0xA5) << np.uint32(24))).view(np.int32)).cuda()
        got = ao.render_batch(dev).cpu().numpy()
        _check_batch(torch, ao, orc, as_float, got, f"D{bits}", as_float=as_float)


@pytest.mark.parametrize("tile", ["0", "1", "2"])
def test_batch_forced_render_tiles(torch_cuda, tile, monkeypatch):
    torch = torch_cuda
    monkeypatch.setenv("MEAO_REN_TILE", tile)
    W, H = 700, 420
    ao, orc = _mk(W, H, intensity=1.1, high_quality_mask=0b0101)
    d = _frames(W, H, 3, seed=31, sky=True)
    got = ao.render_batch(torch.from_numpy(d).cuda()).cpu().numpy()
    _check_batch(torch, ao, orc, d, got, f"MEAO_REN_TILE={tile}", tuple(range(1, 17)) + (18, 20))


@pytest.mark.parametrize("use_graph", [True, False])
def test_batch_forced_tile_loop_and_graph_modes(torch_cuda, use_graph, monkeypatch):
    """The persistent tile loop on every level: the tile cursor runs over all frames, the prefetched next tile may be the next
    frame's.  Three replays: the batch arena's counters must be re-armed each time."""
    torch = torch_cuda
    monkeypatch.setenv("MEAO_UPS_PERSIST_MIN_WAVES", "0.0001")
    W, H = 640, 360
    ao, orc = _mk(W, H, intensity=1.1, high_quality_mask=0b0101, use_graph=use_graph)
    d = _frames(W, H, 3, seed=8, sky=True)
    dd = torch.from_numpy(d).cuda()
    outs = [ao.render_batch(dd).cpu().numpy() for _ in range(3)]
    assert all(np.array_equal(outs[0], o) for o in outs[1:])
    _check_batch(torch, ao, orc, d, outs[0], "forced tile loop", tuple(range(1, 17)) + (18, 20))


def test_batch_graph_reuse_retarget_and_growth(torch_cuda):
    torch = torch_cuda
    W, H = 321, 203
    ao, orc = _mk(W, H, intensity=1.1)
    d5 = torch.from_numpy(_frames(W, H, 5, seed=1)).cuda()
    d2 = torch.from_numpy(_frames(W, H, 2, seed=9)).cuda()
    ref5 = ao.render_batch(d5).clone()
    ref5b = ao.render_batch(d5)                                     # replay of the cached graph
    assert torch.equal(ref5, ref5b)
    other_in, other_out = d5.clone(), torch.empty_like(ref5)       # new pointers: a second graph (or a re-targeted one)
    assert torch.equal(ao.render_batch(other_in, other_out), ref5)
    small = ao.render_batch(d2)                                    # a different B on the same context
    for f in range(2):
        assert torch.equal(small[f], ao.render(d2[f]))
    ao2, _ = _mk(W, H, intensity=1.1)
    a = ao2.render_batch(d2).clone()                               # capacity 2 ...
    b = ao2.render_batch(d5)                                       # ... grows to 5: the old batch graphs are dropped
    assert torch.equal(b, ref5) and torch.equal(ao2.render_batch(d2), a)


def test_batch_unaligned_depth_takes_the_scalar_path(torch_cuda):
    torch = torch_cuda
    W, H = 256, 128
    ao, orc = _mk(W, H, intensity=1.1)
    d = _frames(W, H, 3, seed=4)
    flat = torch.empty(d.size + 1, dtype=torch.float32, device="cuda")
    flat[1:] = torch.from_numpy(d.reshape(-1)).cuda()
    shifted = flat[1:].view(3, H, W)                               # base one element past a 16-byte boundary
    assert shifted.data_ptr() % 16 != 0
    got = ao.render_batch(shifted).cpu().numpy()
    _check_batch(torch, ao, orc, d, got, "unaligned", ids=(1, 2, 10))


def test_batch_64x1080p_equals_render_and_oracle(torch_cuda):
    import bench
    from oracle.oracle import Oracle
    torch = torch_cuda
    W, H, B = 1920, 1080, 64
    host = [bench.make_depth(W, H, f) for f in range(4)]
    depth = torch.stack([torch.roll(torch.from_numpy(host[i % 4]), shifts=29 * (i // 4), dims=1) for i in range(B)]).cuda().contiguous()
    ao, _ = _mk(W, H, intensity=1.1)
    got = ao.render_batch(depth)
    single = torch.empty_like(got)
    for f in range(B):
        ao.render(depth[f], single[f])
    assert torch.equal(got, single)
    orc = Oracle(W, H, threads=8, intensity=1.1)
    for f in (0, 31, 63):
        assert np.array_equal(got[f].cpu().numpy(), orc.run(depth[f].cpu().numpy())), f


def test_batch_8x4k_equals_render_and_oracle(torch_cuda):
    import bench
    from oracle.oracle import Oracle
    torch = torch_cuda
    W, H, B = 3840, 2160, 8
    host = [bench.make_depth(W, H, f) for f in range(2)]
    depth = torch.stack([torch.roll(torch.from_numpy(host[i % 2]), shifts=53 * (i // 2), dims=1) for i in range(B)]).cuda().contiguous()
    ao, _ = _mk(W, H, intensity=1.1)
    got = ao.render_batch(depth)
    for f in range(B):
        assert torch.equal(got[f], ao.render(depth[f])), f
    orc = Oracle(W, H, threads=8, intensity=1.1)
    for f in (0, B - 1):
        assert np.array_equal(got[f].cpu().numpy(), orc.run(depth[f].cpu().numpy())), f


def test_batch_does_not_touch_the_single_frame_state(torch_cuda):
    """render_batch, then render, then render_batch on one context: all right, and debug_buffer shows the single frame."""
    torch = torch_cuda
    W, H = 330, 170
    ao, orc = _mk(W, H, intensity=1.1)
    d = _frames(W, H, 3, seed=12)
    one = _frames(W, H, 1, seed=77)[0]
    dd = torch.from_numpy(d).cuda()
    first = ao.render_batch(dd).cpu().numpy()
    ref_one = orc.run(one)
    assert np.array_equal(ao.render(torch.from_numpy(one).cuda()).cpu().numpy(), ref_one)
    second = ao.render_batch(dd).cpu().numpy()
    assert np.array_equal(first, second)
    for bid in (1, 2, 10, 14, 17):                                 # the single-frame arena still holds the single frame
        got = ao.debug_buffer(bid)
        want = orc.codes(bid) if got.dtype == np.uint8 else orc.buffer(bid).astype(got.dtype)
        assert np.array_equal(got, want), bid
    _check_batch(torch, ao, orc, d, second, "after render")


def test_batch_refusals(torch_cuda):
    import ctypes as C
    from miniengineao_b200 import AmbientOcclusion, Camera
    from miniengineao_b200 import _native as N
    torch = torch_cuda
    W, H = 256, 256
    ao = AmbientOcclusion(Camera(W, H), device=0)
    d = torch.zeros((2, H, W), dtype=torch.float32, device="cuda")
    o = torch.empty((2, H, W), dtype=torch.uint8, device="cuda")
    ao.LateUpdate()
    lib = N.lib()
    assert lib.meao_render_batch(ao._ctx, d.data_ptr(), 0, 0, o.data_ptr(), None) == N.MEAO_ERR_INVALID
    assert lib.meao_render_batch(ao._ctx, d.data_ptr(), 0, 65536, o.data_ptr(), None) == N.MEAO_ERR_INVALID
    assert lib.meao_render_batch(ao._ctx, None, 0, 2, o.data_ptr(), None) == N.MEAO_ERR_INVALID
    assert lib.meao_render_batch(ao._ctx, d.data_ptr(), 7, 2, o.data_ptr(), None) == N.MEAO_ERR_INVALID
    buf = (C.c_uint8 * (W * H))()
    assert lib.meao_get_batch_buffer(ao._ctx, 0, 17, buf, W * H) == N.MEAO_ERR_INVALID
    ao.set_row_band(0, 128, -1, 256)
    assert lib.meao_render_batch(ao._ctx, d.data_ptr(), 0, 2, o.data_ptr(), None) == N.MEAO_ERR_UNSUPPORTED
