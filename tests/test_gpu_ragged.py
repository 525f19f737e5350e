"""GPU (-m gpu): ragged batches - frames of different sizes in one [n, H, W] canvas through resize/pad, the network and
the fused post-processing in one device pass - against the same frames run alone."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import pkg_module

pytestmark = pytest.mark.gpu

# padded (h, w) of the canvas frames: square, landscape, portrait, wide, and a small one (narrow tiles, 8 x 9 maps)
SHAPES = [(368, 368), (368, 496), (496, 368), (368, 552), (64, 72), (120, 96)]


@pytest.fixture(scope="module")
def engine(built, he_sd):
    eng = pkg_module("engine")
    return eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=8, peak_cap=1024,
                          human_cap=2048)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _outs(n, H, W):
    return [torch.empty((n, 38 if k % 2 == 0 else 19, H // 8, W // 8), device="cuda") for k in range(12)]


def _forward_alone(net, frame, mode):
    H, W = frame.shape[:2]
    outs = _outs(1, H, W)
    xd = torch.from_numpy(np.ascontiguousarray(frame[None])).cuda()
    net.forward_u8_ptr(xd.data_ptr(), True, 1, H, W, mode, [o.data_ptr() for o in outs], True, _stream())
    torch.cuda.synchronize()
    return [o[0].cpu() for o in outs]


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "fp32"])
@pytest.mark.parametrize("n", [2, 6])
def test_ragged_maps_bit_identical_to_each_frame_alone(engine, mode, n):
    """n = 2: small plan (narrow tiles, 32-wide n-tiles, PDL); n = 6: large plan (16 x 16 tiles, CTA pairs).  Inside its
    extent every one of the 12 stage outputs of a frame equals that frame run alone, bit for bit; outside it is +0.
    The canvas bytes outside the extents are random: they must not be read."""
    nat = pkg_module("_native")
    shapes = [(368, 496), (64, 72)] if n == 2 else SHAPES
    H, W = max(h for h, _ in shapes), max(w for _, w in shapes)
    rs = np.random.RandomState(100 + n)
    canvas = rs.randint(0, 256, (n, H, W, 3)).astype(np.uint8)
    outs = _outs(n, H, W)
    xd = torch.from_numpy(canvas).cuda()
    engine.net.forward_u8_ragged_ptr(xd.data_ptr(), True, n, H, W, [h for h, _ in shapes], [w for _, w in shapes],
                                     nat.MODES[mode], [o.data_ptr() for o in outs], True, _stream())
    torch.cuda.synchronize()
    outs = [o.cpu() for o in outs]
    for i, (h, w) in enumerate(shapes):
        alone = _forward_alone(engine.net, canvas[i, :h, :w], nat.MODES[mode])
        for k in range(12):
            got = outs[k][i]
            assert torch.equal(got[:, :h // 8, :w // 8], alone[k]), (mode, i, k)
            outside = got.clone()
            outside[:, :h // 8, :w // 8] = 0
            assert not bool((outside.view(torch.int32) != 0).any()), (mode, i, k)      # bits of +0 (-0 is 0x80000000)
    assert any(float(outs[11][i].abs().max()) > 0 for i in range(n))


def _raw_frames(seed, sizes):
    rs = np.random.RandomState(seed)
    return [rs.randint(0, 256, (h, w, 3)).astype(np.uint8) for h, w in sizes]


def _alone_rows(engine, frames, dest_size=368):
    rows = []
    for f in frames:
        engine.infer_raw_async_u8(f.ctypes.data, False, 1, f.shape[0], f.shape[1], dest_size)
        rows.append(engine.fetch_arrays()[0].copy())
    return rows


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_ragged_persons_equal_each_frame_alone(built, he_sd, mode):
    """b200pose_infer_raw_u8_ragged: frames of different source sizes - an exact 2x reduction (INTER_AREA), a frame that
    needs no resize, portrait and landscape - give per frame the person rows of b200pose_infer_raw_u8 on it alone."""
    eng = pkg_module("engine")
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode=mode, batch_cap=8, peak_cap=2048, human_cap=2048)
    # canvas 560 x 1104: a 70 x 138 heat-map plane in shared memory (needs the opt-in beyond 48 KB with the static part)
    frames = _raw_frames(5, [(736, 980), (368, 500), (300, 400), (500, 333), (240, 720)])
    t = pe.infer_raw_ragged_async_u8(frames)
    got = pe.fetch_arrays(ticket=t)
    want = _alone_rows(pe, frames)
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)
    assert sum(len(w) for w in want) > 0


def test_infer_images_ragged_equals_bucketed(engine):
    """About 40 frames of mixed sizes and orientations (several ragged runs of up to batch_cap = 8, two in flight):
    infer_images(ragged=True) == infer_images() frame by frame, rows and normalised dictionaries."""
    rs = np.random.RandomState(11)
    sizes = [(int(rs.randint(100, 420)), int(rs.randint(100, 420))) for _ in range(38)] + [(200, 400), (400, 200)]
    frames = _raw_frames(12, sizes)
    a = engine.infer_images_arrays(frames, dest_size=184)
    b = engine.infer_images_arrays(frames, dest_size=184, ragged=True)
    assert len(a) == len(b) == len(frames)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert sum(len(x) for x in a) > 0
    d = engine.infer_images(frames[:10], dest_size=184, ragged=True)
    assert d == engine.infer_images(frames[:10], dest_size=184)


def test_two_ragged_runs_in_flight(engine):
    """Two ragged runs with different shape sets submitted before either is fetched: each ticket reads its own results
    (per-run extents of the post-processing, per-image normalisation)."""
    fa = _raw_frames(21, [(300, 400), (400, 300), (184, 184)])
    fb = _raw_frames(22, [(200, 600), (250, 250)])
    ta = engine.infer_raw_ragged_async_u8(fa, dest_size=184)
    tb = engine.infer_raw_ragged_async_u8(fb, dest_size=184)
    ra = [r.copy() for r in engine.fetch_arrays(ticket=ta)]
    da = engine.fetch(ticket=ta)
    rb = [r.copy() for r in engine.fetch_arrays(ticket=tb)]
    for got, want in ((ra, _alone_rows(engine, fa, 184)), (rb, _alone_rows(engine, fb, 184))):
        assert len(got) == len(want)
        for g, w in zip(got, want):
            np.testing.assert_array_equal(g, w)
    nat = pkg_module("_native")
    for f, rows, dicts in zip(fa, ra, da):
        _, _, (ph, pw) = nat.crop_geometry(f.shape[0], f.shape[1], 184, 8)
        assert dicts == pkg_module("engine").humans_to_dicts(rows, pw, ph)


def test_ragged_bad_input_raises(engine):
    nat = pkg_module("_native")
    outs = _outs(2, 64, 64)
    xd = torch.zeros((2, 64, 64, 3), dtype=torch.uint8, device="cuda")
    ptrs = [o.data_ptr() for o in outs]
    for eh, ew in (([64, 60], [64, 64]), ([64, 72], [64, 64]), ([0, 64], [64, 64]), ([64, 64], [64, -8])):
        with pytest.raises(nat.B200PoseError, match="extent"):
            engine.net.forward_u8_ragged_ptr(xd.data_ptr(), True, 2, 64, 64, eh, ew, nat.MODE_BF16, ptrs, True, _stream())
    with pytest.raises(nat.B200PoseError):       # more images than the extent array holds (checked before any read)
        engine.net.forward_u8_ragged_ptr(xd.data_ptr(), True, 5000, 8, 8, [8] * 5000, [8] * 5000, nat.MODE_BF16, ptrs,
                                         True, _stream())
    lib = nat.lib()
    assert lib.b200pose_net_forward_u8_ragged(engine.net._h, ctypes.c_void_p(xd.data_ptr()), 1, 2, 64, 64, None, None,
                                              nat.MODE_BF16, None, 1, None) != 0
    frames = _raw_frames(3, [(100, 120)] * 9)
    with pytest.raises(nat.B200PoseError, match="batch_cap"):
        engine.infer_raw_ragged_async_u8(frames)
    with pytest.raises(nat.B200PoseError):
        engine.infer_raw_ragged_async_u8([])
    with pytest.raises(nat.B200PoseError):
        engine.infer_images(frames[:2], ragged=True, flip=True)
    with pytest.raises(nat.B200PoseError):
        engine.infer_images(frames[:2], ragged=True, scales=(0.5, 1.0))
    # the objects are still usable after the rejected calls
    t = engine.infer_raw_ragged_async_u8(frames[:2], dest_size=184)
    got = engine.fetch_arrays(ticket=t)
    for g, w in zip(got, _alone_rows(engine, frames[:2], 184)):
        np.testing.assert_array_equal(g, w)
