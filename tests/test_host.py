"""CPU: host-side logic, the C-ABI surface, and the sequential-exact device cores compiled for the host."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import POST_CASES, ROOT, RecordedPafprocess, assert_humans_equal, golden, pkg_module
from oracle import glue_port, net_port, nms_port, pafprocess_oracle, synth


def test_library_exports_every_declared_symbol(built):
    header = open(os.path.join(ROOT, "include", "b200pose.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\(", header)) - {"defined", "void"}
    nat = pkg_module("_native")
    assert os.path.exists(nat.LIB_PATH)
    lib = ctypes.CDLL(nat.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, "declared in include/b200pose.h but not exported: %s" % missing
    assert set(nat.EXPORTED) <= declared
    assert lib.b200pose_version() == 100
    dims = (ctypes.c_long * 4)()
    assert lib.b200pose_net_tensor_shape(0, dims) == 4 and list(dims) == [64, 3, 3, 3]
    assert lib.b200pose_net_tensor_shape(183, dims) == 1 and dims[0] == 19


def test_no_cpu_fallback(built):
    nat = pkg_module("_native")
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    h = ctypes.c_void_p()
    assert nat.lib().b200pose_net_create(ctypes.byref(h), 0) != 0
    assert b"no CUDA device" in nat.lib().b200pose_last_error()
    model = pkg_module("lib.network.rtpose_vgg").get_model("vgg19")
    with pytest.raises(nat.B200PoseError):
        model(torch.zeros(1, 3, 16, 16))


def test_product_never_touches_the_oracle():
    """The product path must not import / link / execute anything under oracle/ (nor read /root/reference)."""
    pkg = os.path.join(ROOT, "pytorch_realtime_multi-person_pose_estimation_b200")
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|libpafprocess_(port|ref)|oracle[/.](net_port|nms_port|glue_port|synth)"
                     r"|open\(.*/root/reference|sys\.path.*reference", re.M)
    offenders = []
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")) and pat.search(open(os.path.join(d, f), errors="ignore").read()):
                offenders.append(os.path.join(d, f))
    for f in ("lib/__init__.py", "evaluate/__init__.py", "_b200_alias.py"):
        if pat.search(open(os.path.join(ROOT, f)).read()):
            offenders.append(f)
    assert not offenders, offenders


def test_model_has_reference_state_dict_and_loads_strictly(he_sd):
    import lib.network.rtpose_vgg as m        # the reference's import path, aliased to the package
    model = m.get_model("vgg19")
    sd = model.state_dict()
    spec = net_port.state_dict_spec()
    assert list(sd) == list(spec) and all(tuple(sd[k].shape) == spec[k] for k in spec)
    model.load_state_dict(he_sd, strict=True)
    prefixed = {"model." + k: v for k, v in he_sd.items()}       # evaluation.py:13-23 strips a 6-char prefix
    model.load_state_dict({k[6:]: v for k, v in prefixed.items()}, strict=True)
    assert model.float().eval() is model
    with pytest.raises(NotImplementedError):
        m.get_model("mobilenet")


def test_reference_import_paths_resolve():
    from evaluate.coco_eval import get_outputs, handle_paf_and_heat          # noqa: F401
    from lib.config import cfg, update_config
    from lib.network import im_transform
    from lib.pafprocess import pafprocess
    from lib.utils.common import BodyPart, CocoColors, CocoPairsRender, CocoPart, Human, draw_humans  # noqa: F401
    from lib.utils.paf_to_pose import paf_to_pose_cpp                          # noqa: F401
    assert cfg.DATASET.IMAGE_SIZE == 368 and cfg.MODEL.DOWNSAMPLE == 8 and cfg.TEST.THRESH_HEATMAP == 0.1
    class A: cfg = os.path.join(ROOT, "experiments", "vgg19_368x368_sgd.yaml"); opts = ["TEST.THRESH_HEATMAP", "0.2"]
    update_config(cfg, A)
    assert cfg.TEST.THRESH_HEATMAP == 0.2 and cfg.MODEL.NUM_KEYPOINTS == 18
    cfg.defrost(); cfg.TEST.THRESH_HEATMAP = 0.1; cfg.freeze()
    assert all(hasattr(pafprocess, n) for n in ("process_paf", "get_num_humans", "get_part_cid", "get_score",
                                                 "get_part_x", "get_part_y", "get_part_score"))
    assert len(CocoPairsRender) == 17 and CocoPart.Background.value == 18
    img = np.random.RandomState(0).randint(0, 256, (200, 230, 3)).astype(np.uint8)
    a, s, shp = im_transform.crop_with_factor(img, 368, factor=8, is_ceil=True)
    b, s2, shp2 = glue_port.crop_with_factor(img, 368, 8)
    assert a.shape == (368, 424, 3) and s == s2 and shp == shp2
    np.testing.assert_array_equal(a, b)


def test_preprocess_and_flip_match_oracle():
    pre = pkg_module("lib.datasets.preprocessing")
    ev = pkg_module("evaluate.coco_eval")
    img = np.random.RandomState(5).randint(0, 256, (16, 24, 3)).astype(np.uint8)
    np.testing.assert_array_equal(pre.rtpose_preprocess(img), glue_port.rtpose_preprocess(img))
    np.testing.assert_allclose(pre.vgg_preprocess(img), glue_port.vgg_preprocess(img), atol=1e-6)
    rs = np.random.RandomState(6)
    nh, fh, npf, fpf = (rs.rand(6, 5, c).astype(np.float32) for c in (19, 19, 38, 38))
    ap, ah = ev.handle_paf_and_heat(nh.copy(), fh.copy(), npf.copy(), fpf.copy())
    bp, bh = glue_port.handle_paf_and_heat(nh, fh, npf, fpf)
    np.testing.assert_array_equal(ap, bp)
    np.testing.assert_array_equal(ah, bh)


def test_preprocess_device_core_on_host_matches_reference_golden(built):
    """csrc/preprocess_core.h (what conv_first_kernel applies while loading uint8 frames) compiled for the host, the
    product's numpy functions and the reference's own functions (golden) agree bit for bit on every uint8 value, for
    all four `preprocess` modes of get_outputs."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    lib.core_preprocess.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    pre = pkg_module("lib.datasets.preprocessing")
    nat = pkg_module("_native")
    f = golden("preprocess")
    img = np.ascontiguousarray(f["img"])
    for name, fn in (("rtpose", pre.rtpose_preprocess), ("vgg", pre.vgg_preprocess), ("inception", pre.inception_preprocess),
                     ("ssd", pre.ssd_preprocess)):
        out = np.empty((3,) + img.shape[:2], np.float32)
        lib.core_preprocess(nat.PREPROCESS[name], img.ctypes.data, img.shape[0], img.shape[1], out.ctypes.data)
        np.testing.assert_array_equal(out, f[name])
        np.testing.assert_array_equal(fn(img.copy()), f[name])


def _flip_inputs():
    """The seeded inputs tests/golden/make_golden.py fed to the reference's handle_paf_and_heat."""
    return [np.random.RandomState(sd).rand(6, 5, c).astype(np.float32) for sd, c in ((1, 19), (2, 19), (3, 38), (4, 38))]


def test_flip_merge_device_core_on_host_matches_reference_golden(built):
    """csrc/tta_core.h (the functions the CUDA kernel calls) compiled for the host: bit-identical to the reference's
    handle_paf_and_heat golden vector and to the oracle, in both layouts and for a batch."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    lib.core_flip_merge.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 5

    def run(normal, flipped, layout):
        normal, flipped = np.ascontiguousarray(normal), np.ascontiguousarray(flipped)
        out = np.empty_like(normal)
        n, ch = normal.shape[0], (normal.shape[3] if layout == 1 else normal.shape[1])
        h, w = (normal.shape[1:3] if layout == 1 else normal.shape[2:4])
        assert lib.core_flip_merge(normal.ctypes.data, flipped.ctypes.data, out.ctypes.data, n, ch, h, w, layout) == 0
        return out
    nh, fh, npf, fpf = _flip_inputs()
    f = golden("flip_merge")
    np.testing.assert_array_equal(run(nh[None], fh[None], 1)[0], f["avg_heat"])
    np.testing.assert_array_equal(run(npf[None], fpf[None], 1)[0], f["avg_paf"])
    rs = np.random.RandomState(11)
    bnh, bfh, bnp, bfp = (rs.randn(3, 7, 9, c).astype(np.float32) for c in (19, 19, 38, 38))
    for i in range(3):
        ap, ah = glue_port.handle_paf_and_heat(bnh[i], bfh[i], bnp[i], bfp[i])
        np.testing.assert_array_equal(run(bnh, bfh, 1)[i], ah)
        np.testing.assert_array_equal(run(bnp, bfp, 1)[i], ap)
        # NCHW, the layout the fused path merges in
        np.testing.assert_array_equal(run(bnh.transpose(0, 3, 1, 2), bfh.transpose(0, 3, 1, 2), 0)[i], ah.transpose(2, 0, 1))
        np.testing.assert_array_equal(run(bnp.transpose(0, 3, 1, 2), bfp.transpose(0, 3, 1, 2), 0)[i], ap.transpose(2, 0, 1))


def _host_crop(lib, img, dest, factor=8):
    img = np.ascontiguousarray(img)
    g = np.zeros(6)
    lib.core_crop_with_factor(img.ctypes.data, img.shape[0], img.shape[1], dest, factor, None, g.ctypes.data)
    out = np.empty((int(g[3]), int(g[4]), 3), np.uint8)
    lib.core_crop_with_factor(img.ctypes.data, img.shape[0], img.shape[1], dest, factor, out.ctypes.data, g.ctypes.data)
    return out, float(g[0]), (int(g[1]), int(g[2]), 3)


def _core_lib():
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    lib.core_crop_with_factor.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 2
    return lib


def test_crop_with_factor_device_core_on_host_matches_reference_golden_and_cv2(built):
    """csrc/resize_core.h (the functions the CUDA kernel calls) compiled for the host == the reference's
    crop_with_factor golden vectors and == cv2.resize-based oracle on random shapes, bit for bit (incl. the exact-2x
    INTER_AREA switch with a cut last box, up-scaling, 1-pixel-wide frames)."""
    lib = _core_lib()
    f = golden("crop_with_factor")
    for name, h, w, dest, seed in (("50x61", 50, 61, 96, 5), ("64x71_half", 64, 71, 32, 6), ("30x22_up", 30, 22, 40, 7)):
        img = np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)
        out, scale, shape = _host_crop(lib, img, dest)
        np.testing.assert_array_equal(out, f[name + "_out"])
        assert [scale, shape[0], shape[1]] == list(f[name + "_meta"])
    rs = np.random.RandomState(3)
    shapes = [(int(rs.randint(8, 500)), int(rs.randint(8, 500))) for _ in range(40)]
    shapes += [(736, 739), (739, 736), (737, 736), (368, 368), (368, 392), (480, 640), (2, 3), (1, 7), (9, 1)]
    for (h, w) in shapes:
        img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        dest = int(rs.choice([184, 368, 552]))
        want, ws, wshape = glue_port.crop_with_factor(img, dest, 8)
        out, scale, shape = _host_crop(lib, img, dest)
        assert out.shape == want.shape and scale == ws and shape == tuple(wshape), (h, w, dest)
        np.testing.assert_array_equal(out, want)


def test_crop_geometry_and_python_wrappers_without_a_gpu(built, monkeypatch):
    """b200pose_crop_geometry is host arithmetic (callable without a GPU).  The Python wrappers around the device entry
    points (NativeNet.crop_with_factor, PoseEngine.infer_images' shape bucketing) are exercised against a stand-in
    library whose device calls are emulated with the host build of the same core."""
    nat = pkg_module("_native")
    eng = pkg_module("engine")
    for (h, w, dest) in ((200, 230, 368), (368, 368, 368), (736, 739, 368), (1080, 1920, 368), (97, 64, 200)):
        img = np.zeros((h, w, 3), np.uint8)
        want, ws, wshape = glue_port.crop_with_factor(img, dest, 8)
        scale, res, pad = nat.crop_geometry(h, w, dest, 8)
        assert scale == ws and res == tuple(wshape[:2]) and pad == want.shape[:2]
    with pytest.raises(nat.B200PoseError):
        nat.crop_geometry(100, 100, 368, 12)          # factor must be a multiple of the network stride
    core, real = _core_lib(), nat.lib()
    calls = []

    class Fake:
        b200pose_crop_geometry = staticmethod(real.b200pose_crop_geometry)
        b200pose_last_error = staticmethod(real.b200pose_last_error)

        @staticmethod
        def b200pose_net_crop_with_factor(h, images, on_dev, n, sh, sw, dest, factor, out, out_on_dev, stream):
            g = np.zeros(6)
            for i in range(n):
                core.core_crop_with_factor(images.value + i * sh * sw * 3, sh, sw, dest, factor, None, g.ctypes.data)
                core.core_crop_with_factor(images.value + i * sh * sw * 3, sh, sw, dest, factor,
                                           out.value + i * int(g[3]) * int(g[4]) * 3, g.ctypes.data)
            return 0

        @staticmethod
        def b200pose_infer_raw_u8(net, post, images, on_dev, n, sh, sw, dest, factor, mode, thresh, flip, stream):
            first = np.ctypeslib.as_array(ctypes.cast(images.value, ctypes.POINTER(ctypes.c_ubyte)), (n, sh, sw, 3))[:, 0, 0, 0]
            calls.append((n, sh, sw, flip, [int(v) for v in first]))
            return 0

    ms_calls = []

    def fake_multiscale(net, post, images, on_dev, n, sh, sw, base, factor, scales, ns, mode, thresh, flip, stream):
        ms_calls.append((n, sh, sw, base, factor, [scales[i] for i in range(ns)], flip))
        calls.append((n, sh, sw, flip, [0] * n))
        return 0
    Fake.b200pose_infer_raw_u8_multiscale = staticmethod(fake_multiscale)
    monkeypatch.setattr(nat, "lib", lambda: Fake)
    net = object.__new__(eng.NativeNet)
    net._h = None
    rs = np.random.RandomState(8)
    frames = rs.randint(0, 256, (3, 120, 90, 3)).astype(np.uint8)
    out, scale, shape = net.crop_with_factor(frames, 184, 8)
    for i in range(3):
        want, ws, wshape = glue_port.crop_with_factor(frames[i], 184, 8)
        np.testing.assert_array_equal(out[i], want)
        assert scale == ws and shape == tuple(wshape)
    one, _, _ = net.crop_with_factor(frames[1], 184, 8)
    np.testing.assert_array_equal(one, out[1])

    class StubPost:
        batch_cap = 2
        def last_ticket(self): return 0
    pe = object.__new__(eng.PoseEngine)
    pe.net, pe.post, pe.mode = net, StubPost(), 0
    pe.net._h = pe.post._h = None
    pe.fetch = lambda: [("humans-of", v) for v in calls[-1][4]]
    imgs = [np.full((40, 50, 3), 1, np.uint8), np.full((30, 50, 3), 2, np.uint8), np.full((40, 50, 3), 3, np.uint8),
            np.full((40, 50, 3), 4, np.uint8), np.full((30, 50, 3), 5, np.uint8)]
    res = pe.infer_images(imgs, dest_size=64, flip=True)
    assert res == [("humans-of", i + 1) for i in range(5)]                         # input order is restored
    assert [(c[0], c[1], c[2], c[3]) for c in calls] == [(2, 40, 50, 1), (1, 40, 50, 1), (2, 30, 50, 1)]   # <= batch_cap
    assert pe._last == (2, 64, 112)                                               # padded size of the last bucket (30x50 -> 64x107)
    with pytest.raises(nat.B200PoseError):
        pe.infer_images([np.zeros((4, 4), np.uint8)])
    pe.infer_images(imgs[:1], dest_size=64, scales=(0.5, 1.0, 1.5, 2.0), flip=True)
    assert ms_calls == [(1, 40, 50, 64, 8, [0.5, 1.0, 1.5, 2.0], 1)] and pe._last == (1, 64, 80)


def _eval_humans(Human, BodyPart, seed=17, count=5):
    """Same generator as tests/golden/make_golden.py::eval_humans (which fed the reference's append_result)."""
    rs = np.random.RandomState(seed)
    humans = []
    for k in range(count):
        hm = Human([])
        for p in range(18):
            if rs.rand() < 0.75:
                hm.body_parts[p] = BodyPart('%d-%d' % (k, p), p, float(rs.rand()), float(rs.rand()), float(rs.rand()))
        hm.score = float(rs.rand())
        humans.append(hm)
    return humans


def test_append_result_matches_reference_golden():
    """COCO record formatting (coco_eval.py:117-154): 18 -> 17 keypoint reorder, un-scaling, constant score."""
    ev = pkg_module("evaluate.coco_eval")
    common = pkg_module("lib.utils.common")
    f = golden("append_result")
    outputs = []
    ev.append_result(42, _eval_humans(common.Human, common.BodyPart), (368 / 0.71, 496 / 0.71), outputs)
    assert len(outputs) == len(f["keypoints"]) == 5
    for o, kp, sc, iid, cid in zip(outputs, f["keypoints"], f["score"], f["image_id"], f["category_id"]):
        assert list(o.keys()) == list(f["keys"]) and len(o["keypoints"]) == 51
        np.testing.assert_array_equal(np.array(o["keypoints"], np.float64), kp)
        assert o["score"] == sc and o["image_id"] == iid and o["category_id"] == cid


def test_run_eval_plumbing_with_stub_pycocotools(monkeypatch, tmp_path):
    """run_eval (coco_eval.py:245-283) end to end on the host side: image listing, visualisation files, COCO records,
    results.json round trip - with get_outputs / paf_to_pose_cpp (the GPU calls) and pycocotools stubbed."""
    import json
    import types
    import cv2
    ev = pkg_module("evaluate.coco_eval")
    common = pkg_module("lib.utils.common")
    img_dir, vis_dir = tmp_path / "img", tmp_path / "vis"
    img_dir.mkdir(); vis_dir.mkdir()
    rs = np.random.RandomState(2)
    for name, shape in (("a.jpg", (60, 80, 3)), ("b.jpg", (90, 70, 3))):
        cv2.imwrite(str(img_dir / name), rs.randint(0, 256, shape).astype(np.uint8))
    seen = {}

    class COCO:
        def __init__(self, anno): seen["anno"] = anno
        def getCatIds(self, catNms): return [1]
        def getImgIds(self, catIds): return [7, 9]
        def loadImgs(self, i): return [{"file_name": {7: "a.jpg", 9: "b.jpg"}[i]}]
        def loadRes(self, path): seen["results"] = json.load(open(path)); return "dt"

    class COCOeval:
        def __init__(self, gt, dt, kind): self.params = types.SimpleNamespace(imgIds=None); self.stats = [0.5]; seen["kind"] = kind
        def evaluate(self): seen["imgIds"] = self.params.imgIds
        def accumulate(self): pass
        def summarize(self): pass
    for name, attrs in (("pycocotools", {}), ("pycocotools.coco", {"COCO": COCO}), ("pycocotools.cocoeval", {"COCOeval": COCOeval})):
        m = types.ModuleType(name); m.__dict__.update(attrs); monkeypatch.setitem(sys.modules, name, m)
    humans = _eval_humans(common.Human, common.BodyPart, seed=3, count=2)
    monkeypatch.setattr(ev, "get_outputs", lambda img, model, pre: (np.zeros((46, 62, 38), np.float32),
                                                                    np.zeros((46, 62, 19), np.float32), 368.0 / min(img.shape[:2])))
    monkeypatch.setattr(ev, "paf_to_pose_cpp", lambda heat, paf, cfg: humans)
    monkeypatch.chdir(tmp_path)
    assert ev.run_eval(str(img_dir), "anno.json", str(vis_dir), model=None, preprocess="rtpose") == 0.5
    assert sorted(os.listdir(vis_dir)) == ["a.jpg", "b.jpg"] and not os.path.exists(tmp_path / "results.json")
    assert seen["kind"] == "keypoints" and seen["imgIds"] == [7, 9] and len(seen["results"]) == 4
    want = []
    ev.append_result(7, humans, (46 * 8 / (368.0 / 60), 62 * 8 / (368.0 / 60)), want)
    assert seen["results"][:2] == json.loads(json.dumps(want))
    # the import-compatibility surface of evaluate/evaluation.py:4-7
    from evaluate.coco_eval import run_eval                                   # noqa: F401
    from lib.network.openpose import OpenPose_Model, use_vgg                  # noqa: F401
    from lib.network.rtpose_vgg import get_model, use_vgg as use_vgg2         # noqa: F401
    with pytest.raises(NotImplementedError):
        OpenPose_Model(l2_stages=4, l1_stages=2, paf_out_channels=38, heat_out_channels=19)


def test_cubic_resize_device_core_on_host_matches_oracle(built):
    """csrc/resize_core.h rs_cubic_* (the functions resize_cubic_accum_kernel calls) compiled for the host == the
    oracle's restatement of OpenCV's INTER_CUBIC, bit for bit, for the size ratios of the multi-scale averaging."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    lib.core_resize_cubic.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 3 + [ctypes.c_void_p] + [ctypes.c_int] * 2
    rs = np.random.RandomState(13)
    cases = [(23, 23, 46, 46, 19), (69, 69, 46, 46, 38), (92, 92, 46, 46, 19), (6, 9, 12, 16, 38), (24, 33, 12, 16, 19),
             (46, 53, 46, 53, 38), (1, 1, 4, 4, 19), (2, 1, 3, 5, 38), (1, 7, 9, 2, 1)] + \
            [tuple(int(v) for v in rs.randint(3, 80, 4)) + (int(rs.choice([1, 19, 38])),) for _ in range(20)]
    for (h, w, dh, dw, c) in cases:
        src = rs.randn(h, w, c).astype(np.float32)
        out = np.empty((dh, dw, c), np.float32)
        lib.core_resize_cubic(src.ctypes.data, h, w, c, out.ctypes.data, dh, dw)
        np.testing.assert_array_equal(out, glue_port.resize_cubic(src, dh, dw))


@pytest.mark.parametrize("name", sorted(POST_CASES))
def test_device_cores_on_host_match_oracle(name, built):
    """csrc/post_core.h (pair scoring, std::sort emulation, greedy matching, indexed person assembly) compiled
    for the host must reproduce the oracle exactly - same code the CUDA kernels execute."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    FP = ctypes.POINTER(ctypes.c_float)
    lib.core_process.argtypes = [ctypes.c_int, FP, ctypes.c_int, FP, ctypes.c_long, ctypes.c_long, ctypes.c_long,
                                 ctypes.c_int, ctypes.c_int]
    lib.core_result.restype = FP
    heat, paf = POST_CASES[name](synth)
    h, w = heat.shape[:2]
    jl, want = glue_port.paf_to_pose(heat, paf, pafprocess_oracle.load_port())
    jl = np.ascontiguousarray(jl)
    paf = np.ascontiguousarray(paf)
    nh = lib.core_process(len(jl), jl.ctypes.data_as(FP), h * 8, paf.ctypes.data_as(FP), 1, w * 38, 38, 3, 0)
    rows = (np.ctypeslib.as_array(lib.core_result(), shape=(nh * 73,)).reshape(nh, 73) if nh else
            np.zeros((0, 73), np.float32))
    got = pkg_module("engine").humans_to_dicts(rows, w * 8, h * 8)
    assert_humans_equal(got, want, score_tol=0.0)
    assert lib.core_sort_mismatch() == 0      # warp-chunked partition == sequential std::sort emulation


def test_device_cores_on_host_fuzz_against_the_compiled_reference(built):
    """300 random pafprocess inputs (peak sets with clusters / duplicated pixels, direction fields with exact ties, person
    shapes with cross links) through csrc/post_core.h on the host, against what the reference's own pafprocess.cpp
    returned on them (golden): identical persons, scores and part assignments."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    FP = ctypes.POINTER(ctypes.c_float)
    lib.core_process.argtypes = [ctypes.c_int, FP, ctypes.c_int, FP, ctypes.c_long, ctypes.c_long, ctypes.c_long,
                                 ctypes.c_int, ctypes.c_int]
    lib.core_result.restype = FP
    ref = RecordedPafprocess()
    to_dicts = pkg_module("engine").humans_to_dicts

    def ref_humans(t, jl, paf, h, w):
        ref.select(t, jl, paf)
        out = []
        for hid in range(ref.get_num_humans()):
            parts = {}
            for p in range(18):
                c = int(ref.get_part_cid(hid, p))
                if c >= 0:
                    parts[p] = (float(ref.get_part_x(c)) / (w * 8), float(ref.get_part_y(c)) / (h * 8),
                                float(ref.get_part_score(c)))
            if parts:
                out.append((float(ref.get_score(hid)), parts))
        return out
    humans = 0
    for t in range(300):
        h, w, jl, paf = synth.fuzz_scenario(t)
        if len(jl) == 0:
            continue
        want = ref_humans(t, jl, paf, h, w)
        nh = lib.core_process(len(jl), jl.ctypes.data_as(FP), h * 8, paf.ctypes.data_as(FP), 1, w * 38, 38, 3, 0)
        rows = (np.ctypeslib.as_array(lib.core_result(), shape=(nh * 73,)).reshape(nh, 73).copy() if nh else
                np.zeros((0, 73), np.float32))
        assert to_dicts(rows, w * 8, h * 8) == want, "scenario seed %d" % (1000 + t)
        assert lib.core_sort_mismatch() == 0
        humans += len(want)
    assert humans > 300


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    import _b200_alias
    _b200_alias.load_package()
    import importlib
    dist_mod = importlib.import_module(_b200_alias.PKG + ".distributed")
    sd = net_port.he_state_dict(1234) if rank == 0 else None
    arrays = dist_mod.broadcast_state_arrays([v.numpy() for v in sd.values()] if sd else None, device="cpu")
    lo, hi = dist_mod.shard_range(67, rank, world)
    q.put((rank, lo, hi, float(sum(float(a.sum()) for a in arrays[:6])), len(arrays)))
    dist.destroy_process_group()


def test_multi_gpu_host_logic_with_gloo():
    """world_size-2 gloo: weights are broadcast once from rank 0, frames shard contiguously, no other collective."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=180) for _ in procs)
    [p.join(timeout=60) for p in procs]
    assert res[0][1:3] == (0, 34) and res[1][1:3] == (34, 67)
    assert res[0][3] == res[1][3] and res[0][4] == res[1][4] == 184


def test_warp_partition_reproduces_std_sort(built):
    """The chunked (32-wide) Hoare partition the GPU runs gives the same permutation as the sequential libstdc++
    introsort restatement, including the order of equal keys, on duplicate-heavy and adversarial inputs."""
    lib = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    U = ctypes.POINTER(ctypes.c_uint64)
    lib.core_sort_check.argtypes = [U, ctypes.c_int, U]
    rs = np.random.RandomState(0)
    def check(hi):
        n = len(hi)
        keys = (hi.astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)
        out = np.zeros(max(n, 1), np.uint64)
        assert lib.core_sort_check(keys.ctypes.data_as(U), n, out.ctypes.data_as(U)) == 0
        out = out[:n]
        assert np.all((out[:-1] >> np.uint64(32)) <= (out[1:] >> np.uint64(32)))
        assert sorted(out.tolist()) == sorted(keys.tolist())
    for n in list(range(0, 40)) + [63, 64, 65, 100, 257, 1000, 4097, 30000]:
        for distinct in (1, 2, 7, max(1, n // 3), 1 << 30):
            check(rs.randint(0, distinct, size=n))
    for n in (17, 33, 100, 1000, 5000):
        for hi in (np.arange(n), np.arange(n)[::-1], np.minimum(np.arange(n), np.arange(n)[::-1]), np.arange(n) % 2,
                   np.arange(n) % 17):
            check(np.ascontiguousarray(hi))


def test_data_parallel_replica_finds_the_master_weights(he_sd):
    """torch.nn.parallel.replicate builds shallow copies whose `_parameters` are EMPTY; rtpose_model must take its
    weights and its engine cache from the module that owns them (ADVICE r1: IndexError in _signature on a replica)."""
    import copy
    import pickle
    import lib.network.rtpose_vgg as m
    model = m.get_model("vgg19")
    model.load_state_dict(he_sd)

    def replica_of(mod):          # what replicate() leaves behind, minus the device copies
        rep = mod._replicate_for_data_parallel()
        for name, child in mod._modules.items():
            rep._modules[name] = replica_of(child)
        return rep
    rep = replica_of(model)
    assert len(list(rep.parameters())) == 0 and len(rep.state_dict()) == 0
    assert rep._master[0] is model and rep._engines is model._engines
    assert len(rep._master[0]._signature()) == 184
    # the signature covers every tensor: an in-place edit of any of them invalidates the packed device copy
    before = model._signature()
    with torch.no_grad():
        list(model.parameters())[101].mul_(1.0)
    assert model._signature() != before
    # copies own their state
    c = copy.deepcopy(model)
    assert c._master[0] is c and c._engines is not model._engines and len(c.state_dict()) == 184
    d = pickle.loads(pickle.dumps(model))
    assert d._master[0] is d and torch.equal(d.state_dict()["model0.0.weight"], he_sd["model0.0.weight"])


def test_engine_remembers_the_shape_of_each_ticket(built):
    """Two runs in flight with different batch sizes / frame shapes: fetch(ticket=i) must use run i's (n, H, W)
    (ADVICE r1).  Pure host logic, exercised on an engine object without native handles."""
    eng = pkg_module("engine")
    nat = pkg_module("_native")
    pe = object.__new__(eng.PoseEngine)
    pe._shapes, pe._last = {}, None

    class FakePost:
        t = -1

        def last_ticket(self):
            return self.t
    pe.post = FakePost()
    for t, shape in enumerate([(4, 368, 368), (1, 184, 248), (2, 368, 392)]):
        pe.post.t = t
        assert pe._remember(*shape) == t
    assert pe._shape_of(None) == (2, 368, 392) and pe._shape_of(2) == (2, 368, 392) and pe._shape_of(1) == (1, 184, 248)
    with pytest.raises(nat.B200PoseError):
        pe._shape_of(0)          # only the last two runs are retained, like the native result slots


def test_pose_stream_pipelines_two_batches(built):
    """streaming.PoseStream (SURVEY.md 8f rank 4): frames are grouped into batches, batch i+1 is SUBMITTED before batch
    i is fetched (two runs in flight), results come back in frame order, a trailing partial batch is flushed, frames of
    different shapes are refused.  Host logic, exercised with a stand-in engine."""
    streaming = pkg_module("streaming")
    nat = pkg_module("_native")
    log = []

    class FakeNet:
        def set_preprocess(self, name): log.append(("pre", name))

    class FakeEngine:
        net = FakeNet()
        t = -1

        def submit_images(self, images, dest, factor, thresh):
            self.t += 1
            log.append(("submit", self.t, [int(f[0, 0, 0]) for f in images]))
            self.last = {self.t: len(images)}
            FakeEngine.sizes[self.t] = [int(f[0, 0, 0]) for f in images]
            return self.t

        def fetch_arrays(self, ticket=None):
            log.append(("fetch", ticket))
            rows = []
            for v in FakeEngine.sizes[ticket]:      # one person per frame whose nose x encodes the frame's value
                r = np.full((1, 73), -1.0, np.float32)
                r[0, 0] = 1.0
                r[0, 1:5] = (v, 2 * v, 0.5, 0)
                rows.append(r)
            return rows
    FakeEngine.sizes = {}

    class FakeModel:
        def pose_engine(self, batch_cap): log.append(("engine", batch_cap)); return FakeEngine()
    frames = [np.full((48, 64, 3), i, np.uint8) for i in range(7)]
    got = list(streaming.PoseStream(FakeModel(), frames, batch=3, draw=False))
    assert [int(f[0, 0, 0]) for f, _, _ in got] == list(range(7))
    _, _, (ph, pw) = nat.crop_geometry(48, 64, 368, 8)       # coordinates are normalised by the padded network input
    assert (ph, pw) == (368, 496)
    assert [h[0].body_parts[0].x for _, h, _ in got] == [float(np.float32(i)) / pw for i in range(7)]
    ops = [e[:2] for e in log if e[0] in ("submit", "fetch")]
    assert ops == [("submit", 0), ("submit", 1), ("fetch", 0), ("submit", 2), ("fetch", 1), ("fetch", 2)]
    assert log[0] == ("engine", 3) and log[1] == ("pre", "rtpose")
    with pytest.raises(nat.B200PoseError):
        list(streaming.PoseStream(FakeModel(), [frames[0], np.zeros((50, 64, 3), np.uint8)], batch=2, draw=False))
    with pytest.raises(nat.B200PoseError):
        streaming.PoseStream(object(), frames)


def test_bench_clock_sampler_keeps_only_rows_inside_the_timed_region():
    """bench.py's clock record must describe the TIMED region: rows of the nvidia-smi poller (started ahead of the
    warm-up) are filtered by their time stamps; with no row inside the window the nearest one is used and named; the
    roofline denominator follows the record (burst only at full clock without a power cap)."""
    import datetime
    import importlib.util
    import time
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class Done:     # stands for the poller process
        def terminate(self): pass
        def wait(self, timeout=None): pass
        def kill(self): pass

    def sampler_with(rows, t0):
        s = bench.ClockSampler(0, None)
        if s.p is not None:
            s.p.kill()
        s.p, s.nv_handle, s.nv_rows = Done(), None, []
        with open(s.f.name, "w") as f:
            for dt_ms, mhz, cap in rows:
                ts = (t0 + datetime.timedelta(milliseconds=dt_ms)).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
                f.write("%s, %d, 1965, 250.5, 0x0, Not Active, Not Active, Not Active, %s\n"
                        % (ts, mhz, "Active" if cap else "Not Active"))
        s.t0 = t0
        return s

    now = datetime.datetime.now()
    s = sampler_with([(-300, 1200, True), (-100, 1500, True), (50, 1965, False), (150, 1965, False), (9000, 900, True)], now)
    time.sleep(0.25)
    rec = s.stop()
    assert rec["samples"] == 2 and rec["sm_mhz"] == 1965.0 and rec["reasons"] == [] and "inside" in rec["source"]
    assert "burst" in bench.peaks(rec)[2]
    s = sampler_with([(-400, 1500, True)], datetime.datetime.now())
    rec = s.stop()
    assert rec["samples"] == 1 and rec["reasons"] == ["sw_power_cap"] and "nearest" in rec["source"]
    assert "sustained" in bench.peaks(rec)[2] and "sustained" in bench.peaks(None)[2]
