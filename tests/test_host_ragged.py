"""CPU: host side of ragged batches (frames of different sizes in one device pass) - the run grouping of
PoseEngine.infer_images(ragged=True), the per-frame crop geometry, and the build of the masked conv kernels."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, pkg_module
from oracle import glue_port


def _random_pads(rs, n):
    nat = pkg_module("_native")
    sizes = [(int(rs.randint(60, 900)), int(rs.randint(60, 900))) for _ in range(n)]
    return [nat.crop_geometry(h, w, 368, 8)[2] for h, w in sizes]


@pytest.mark.parametrize("seed,n,cap", [(0, 1, 32), (1, 40, 8), (2, 257, 32), (3, 64, 1), (4, 33, 32)])
def test_ragged_groups_partition_orientation_cap_canvas(built, seed, n, cap):
    eng = pkg_module("engine")
    pads = _random_pads(np.random.RandomState(seed), n)
    runs = eng.ragged_groups(pads, cap)
    order = [i for part, _ in runs for i in part]
    assert sorted(order) == list(range(n))                          # every frame in exactly one run
    for part, (ch, cw) in runs:
        assert 1 <= len(part) <= cap
        land = {pads[i][0] <= pads[i][1] for i in part}
        assert len(land) == 1                                       # one orientation per run
        assert ch == max(pads[i][0] for i in part) and cw == max(pads[i][1] for i in part)
        long_side = [max(pads[i]) for i in part]
        assert long_side == sorted(long_side)
    assert eng.ragged_groups(pads, cap) == runs                     # deterministic
    inv = np.empty(n, np.int64)
    inv[np.asarray(order)] = np.arange(n)
    assert [order[k] for k in inv] == list(range(n))                # the inverse permutation restores input order


def test_ragged_groups_fill_runs():
    eng = pkg_module("engine")
    pads = [(368, 496)] * 5 + [(496, 368)] * 3 + [(368, 368)] * 2
    runs = eng.ragged_groups(pads, 4)
    assert [len(p) for p, _ in runs] == [4, 3, 3]
    assert [c for _, c in runs] == [(368, 496), (368, 496), (496, 368)]
    assert runs[0][0] == [8, 9, 0, 1]                               # square frames first (shortest long side)
    with pytest.raises(pkg_module("_native").B200PoseError):
        eng.ragged_groups(pads, 0)


RAGGED_SRC = [(480, 640), (640, 480), (427, 640), (612, 612), (375, 500), (736, 980), (368, 500), (241, 719), (720, 240),
              (8, 9)]


@pytest.mark.parametrize("dest_size,factor", [(368, 8), (184, 16)])
def test_ragged_layout_per_frame_geometry_offsets_canvas(built, dest_size, factor):
    """b200pose_ragged_layout - the per-frame geometry b200pose_infer_raw_u8_ragged uses: every frame gets the padded
    size crop_with_factor gives it alone (exact 2x INTER_AREA and no-resize frames included), its byte offset in the
    packed input is the sum of the frames before it, and the canvas is the largest padded height x width."""
    nat = pkg_module("_native")
    off, pads, canvas = nat.ragged_layout(RAGGED_SRC, dest_size, factor)
    assert off == [int(v) for v in np.concatenate([[0], np.cumsum([3 * h * w for h, w in RAGGED_SRC])[:-1]])]
    for (h, w), (ph, pw) in zip(RAGGED_SRC, pads):
        assert (ph, pw) == nat.crop_geometry(h, w, dest_size, factor)[2]
        im = np.random.RandomState(h * 1000 + w).randint(0, 256, (h, w, 3)).astype(np.uint8)
        crop, _, _ = glue_port.crop_with_factor(im, dest_size, factor)
        assert (ph, pw) == crop.shape[:2] and ph % 8 == 0 and pw % 8 == 0
    assert canvas == (max(p[0] for p in pads), max(p[1] for p in pads))
    assert nat.ragged_layout(RAGGED_SRC[4:5], dest_size, factor) == ([0], pads[4:5], pads[4])


def test_ragged_layout_rejects_bad_frames(built):
    nat = pkg_module("_native")
    with pytest.raises(nat.B200PoseError, match="no frames"):
        nat.ragged_layout([])
    with pytest.raises(nat.B200PoseError, match="frame 1"):
        nat.ragged_layout([(100, 120), (0, 50)])
    with pytest.raises(nat.B200PoseError, match="factor"):
        nat.ragged_layout([(100, 120)], 368, 12)


def test_forward_u8_ragged_ptr_checks_extent_lengths(built):
    eng = pkg_module("engine")
    nat = pkg_module("_native")
    net = object.__new__(eng.NativeNet)
    net._h = None
    for eh, ew in (([64, 64, 64], [64, 64]), ([64], [64, 64])):
        with pytest.raises(nat.B200PoseError, match="extents"):
            net.forward_u8_ragged_ptr(0, True, 2, 64, 64, eh, ew, nat.MODE_BF16, [0] * 12, True, 0)


def test_masked_conv_kernels_still_use_tcgen05(built):
    """The extent masking lives in the epilogues: all four tensor-core conv kernels still issue UTCHMMA."""
    lib = os.path.join(ROOT, "pytorch_realtime_multi-person_pose_estimation_b200", "libb200pose.so")
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc")) or "/usr/local/cuda/bin/nvcc"
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(nvcc), "cuobjdump")
    r = subprocess.run([cuobjdump, "-sass", lib], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-2000:]
    funcs = re.split(r"\n\s*Function : ", r.stdout)
    seen = {}
    for f in funcs[1:]:
        name = f.split("\n", 1)[0]
        m = re.search(r"(conv_tc_(?:pair_chunk|pair|chunk)?_?kernel)", name)
        if m:
            seen[m.group(1)] = "UTCHMMA" in f or "UTCQMMA" in f
    assert set(seen) == {"conv_tc_kernel", "conv_tc_pair_kernel", "conv_tc_chunk_kernel", "conv_tc_pair_chunk_kernel"}, seen
    assert all(seen.values()), seen
