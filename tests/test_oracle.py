"""CPU: pins the oracle (CPU restatements under oracle/) against golden vectors produced by the unmodified
reference and its compiled pafprocess.cpp (tests/golden/make_golden.py)."""
import hashlib
import itertools

import numpy as np
import pytest
import torch

from conftest import POST_CASES, assert_humans_equal, golden, humans_rows_to_dicts
from oracle import glue_port, net_exact, net_port, nms_port, pafprocess_oracle, synth


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


@pytest.mark.parametrize("name", ["net_64", "net_368"])
def test_exact_order_network_is_pinned_to_the_reference(name, he_sd):
    """oracle/conv_exact.c (fp32 fused multiply-adds in a defined order) vs the output of the unmodified reference
    module: a different but equally valid fp32 summation order, so the two agree to a few 1e-5 on O(1) maps."""
    g = golden(name)
    hw, seed = int(g["hw"]), int(g["seed"])
    x = torch.rand((1, 3, hw, hw), generator=torch.Generator().manual_seed(seed)) - 0.5
    (paf, heat), saved = net_exact.forward(he_sd, x.numpy())
    assert len(saved) == 12 and paf.shape == g["paf"].shape
    assert np.abs(paf - g["paf"]).max() < 1e-4 and np.abs(heat - g["heat"]).max() < 1e-4
    np.testing.assert_allclose([float(np.abs(t).max()) for t in saved], g["stage_absmax"], rtol=1e-4)


def test_exact_order_network_is_deterministic_and_thread_count_independent(he_sd, monkeypatch):
    x = (torch.rand((2, 3, 40, 56), generator=torch.Generator().manual_seed(2)) - 0.5).numpy()
    _, a = net_exact.forward(he_sd, x)
    monkeypatch.setenv("ORACLE_THREADS", "1")
    _, b = net_exact.forward(he_sd, x)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v)
    # image rows of a batch are independent
    _, c = net_exact.forward(he_sd, x[1:2])
    np.testing.assert_array_equal(c[-1][0], a[-1][1])


@pytest.mark.parametrize("name", ["net_64", "net_368"])
def test_net_port_matches_reference_module(name, he_sd):
    g = golden(name)
    hw, seed = int(g["hw"]), int(g["seed"])
    x = torch.rand((1, 3, hw, hw), generator=torch.Generator().manual_seed(seed)) - 0.5
    assert _digest(x.numpy()) == str(g["x_digest"]), "input regeneration drifted"
    with torch.no_grad():
        (paf, heat), saved = net_port.forward(he_sd, x)
    assert len(saved) == 12
    # same torch ops in the same order as the reference module -> identical up to oneDNN blocking choices
    assert np.abs(paf.numpy() - g["paf"]).max() < 1e-5
    assert np.abs(heat.numpy() - g["heat"]).max() < 1e-5
    np.testing.assert_allclose([float(t.abs().max()) for t in saved], g["stage_absmax"], rtol=1e-5)
    np.testing.assert_allclose(np.stack([t.numpy().reshape(-1)[::13][:64] for t in saved]), g["stage_sample"], atol=1e-5)
    assert float(paf.abs().max()) > 0.5          # non-vacuous: He weights give O(1) outputs


def test_state_dict_spec_is_the_reference_layout():
    spec = net_port.state_dict_spec()
    assert len(spec) == 184
    assert sum(int(np.prod(s)) for s in spec.values()) == 52311446      # SURVEY.md N1
    assert list(spec)[:2] == ["model0.0.weight", "model0.0.bias"] and list(spec)[-1] == "model6_2.12.bias"
    assert spec["model2_1.0.weight"] == (128, 185, 7, 7) and spec["model1_2.8.weight"] == (19, 512, 1, 1)


def test_get_outputs_and_flip_merge(he_sd):
    g = golden("get_outputs_200x230")
    img = np.random.RandomState(0).randint(0, 256, (200, 230, 3)).astype(np.uint8)
    assert _digest(img) == str(g["img_digest"])
    paf, heat, scale = glue_port.get_outputs(img, he_sd, "rtpose")
    assert paf.shape == g["paf"].shape == (46, 53, 38) and abs(scale - float(g["scale"])) < 1e-12
    assert np.abs(paf - g["paf"]).max() < 1e-5 and np.abs(heat - g["heat"]).max() < 1e-5
    f = golden("flip_merge")
    nh, fh = np.random.RandomState(1).rand(6, 5, 19).astype(np.float32), np.random.RandomState(2).rand(6, 5, 19).astype(np.float32)
    npf, fpf = np.random.RandomState(3).rand(6, 5, 38).astype(np.float32), np.random.RandomState(4).rand(6, 5, 38).astype(np.float32)
    ap, ah = glue_port.handle_paf_and_heat(nh, fh, npf, fpf)
    np.testing.assert_array_equal(ap, f["avg_paf"])
    np.testing.assert_array_equal(ah, f["avg_heat"])


def test_bicubic_is_bit_exact_with_opencv_native_path():
    import cv2
    rs = np.random.RandomState(0)
    prev = cv2.ipp.useIPP()
    try:
        for (h, w) in itertools.product([3, 4, 5], [3, 4, 5]):
            for _ in range(4):
                p = rs.rand(h, w).astype(np.float32)
                mine = nms_port.upsample8_cubic(p)
                cv2.ipp.setUseIPP(False)     # OpenCV's own resize.cpp arithmetic
                native = cv2.resize(p, None, fx=8, fy=8, interpolation=cv2.INTER_CUBIC)
                cv2.ipp.setUseIPP(prev)      # the build default (IPP): proprietary arithmetic, a few ulp away
                default = cv2.resize(p, None, fx=8, fy=8, interpolation=cv2.INTER_CUBIC)
                np.testing.assert_array_equal(mine, native)
                assert np.abs(mine - default).max() <= 5e-7
                assert mine.argmax() == default.argmax()
    finally:
        cv2.ipp.setUseIPP(prev)


@pytest.mark.parametrize("name", sorted(POST_CASES))
def test_nms_port_matches_reference_nms(name):
    g = golden("post_" + name)
    heat, paf = POST_CASES[name](synth)
    assert _digest(heat, paf) == str(g["in_digest"]), "synthetic input drifted"
    jl = nms_port.joint_list_from_nms(nms_port.nms(heat, 0.1))
    ref = g["joint_list"]
    assert jl.shape == ref.shape
    if len(jl):
        np.testing.assert_array_equal(jl[:, [0, 1, 3, 4]], ref[:, [0, 1, 3, 4]])   # coordinates, ids, parts: exact
        assert np.abs(jl[:, 2] - ref[:, 2]).max() <= 5e-7                           # scores: IPP vs native cubic


@pytest.mark.parametrize("name", sorted(POST_CASES))
def test_pafprocess_port_matches_reference(name, built):
    g = golden("post_" + name)
    heat, paf = POST_CASES[name](synth)
    port = pafprocess_oracle.load_port()
    _, humans = glue_port.paf_to_pose(heat, paf, port)
    assert_humans_equal(humans, humans_rows_to_dicts(g["humans"]), score_tol=1e-6)
    # the reference's own translation unit on the same peaks (golden) -> bit-identical
    assert humans == humans_rows_to_dicts(golden("pafprocess_ref")["post_" + name])


def test_pafprocess_port_ties_and_scale(built):
    """Large crowded scenes produce exactly-equal candidate scores; std::sort's order is reproduced (golden: the
    reference's own pafprocess.cpp on the same scenes)."""
    port, ref = pafprocess_oracle.load_port(), golden("pafprocess_ref")
    for persons, seed in [(30, 31), (50, 5), (80, 7)]:
        heat, paf, _ = synth.stick_figures(persons, seed)
        a = glue_port.paf_to_pose(heat, paf, port)[1]
        b = humans_rows_to_dicts(ref["ties_%d_%d" % (persons, seed)])
        assert a == b and len(a) > persons // 2


def test_swig_typemap_errors(built):
    port = pafprocess_oracle.load_port()
    with pytest.raises(TypeError):
        port.process_paf(np.zeros((1, 1, 5), np.float64), np.zeros((8, 8, 19), np.float32), np.zeros((8, 8, 38), np.float32))


def test_cubic_resize_restatement_vs_opencv():
    """oracle/glue_port.resize_cubic (the composition oracle of the multi-scale averaging) against cv2.resize
    INTER_CUBIC: within 3e-7 of OpenCV's own code path (IPP off; cv2 evaluates the last row_length % 4 elements of a row
    in another order), identity for equal sizes, exact when the row length is a multiple of 4."""
    import cv2
    rs = np.random.RandomState(12)
    prev = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        for (h, w, dh, dw, c) in ((23, 23, 46, 46, 19), (69, 69, 46, 46, 38), (92, 92, 46, 46, 19), (6, 9, 12, 16, 38),
                                  (24, 33, 12, 16, 19), (46, 53, 46, 53, 19), (20, 30, 33, 47, 1)):
            src = rs.randn(h, w, c).astype(np.float32)
            ref = cv2.resize(src, (dw, dh), interpolation=cv2.INTER_CUBIC).reshape(dh, dw, c)
            mine = glue_port.resize_cubic(src, dh, dw)
            assert np.abs(mine - ref).max() <= 3e-7
            if (dw * c) % 4 == 0 or (h, w) == (dh, dw):
                np.testing.assert_array_equal(mine, ref)
    finally:
        cv2.ipp.setUseIPP(prev)
    x = rs.randn(46, 46, 19).astype(np.float32)
    np.testing.assert_array_equal(glue_port.resize_cubic(x, 46, 46), x)
    h1, p1 = rs.randn(12, 16, 19).astype(np.float32), rs.randn(12, 16, 38).astype(np.float32)
    ah, ap = glue_port.multi_scale_maps([(h1, p1)] * 4, (12, 16))
    np.testing.assert_array_equal(ah, h1)          # (4 x) / 4 is exact
    np.testing.assert_array_equal(ap, p1)
