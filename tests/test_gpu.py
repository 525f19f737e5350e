"""GPU (-m gpu): parity of the CUDA path, called through the C ABI / the reference-shaped Python surface, against
the oracle (CPU) on seeded inputs and against the committed golden vectors of the reference."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import POST_CASES, ROOT, assert_humans_equal, golden, humans_rows_to_dicts, pkg_module
from oracle import glue_port, net_exact, net_port, nms_port, pafprocess_oracle, synth

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-3          # BASELINE.json north_star: heat/PAF within 1e-3 max-abs in fp32 (mode "fp32")
BF16X3_TOL = 1e-3        # the same bar for the tensor-core mode: hi+lo bf16 planes, K-chunked accumulation (measured 1.4e-4
                         # @368x368; 1.4e-3 when the tensor core accumulates all of K = 6272 by itself)
BF16_TOL = 0.15          # bf16 operands through 52 conv layers, outputs O(1..4); measured value is printed


@pytest.fixture(scope="module")
def native_net(built, he_sd):
    eng = pkg_module("engine")
    net = eng.NativeNet(0)
    net.load_state_dict_arrays([v.numpy() for v in he_sd.values()])
    return net


def _forward(net, x, mode):
    nat = pkg_module("_native")
    n, _, H, W = x.shape
    outs = [torch.empty((n, 38 if i % 2 == 0 else 19, H // 8, W // 8), device="cuda") for i in range(12)]
    xd = x.cuda().contiguous()
    net.forward_ptr(xd.data_ptr(), True, n, H, W, nat.MODES[mode], [o.data_ptr() for o in outs], True,
                    torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return [o.cpu() for o in outs]


def test_tcgen05_conv_kernel_cases(built):
    """Standalone harness: 7 conv configurations (1x1/3x3/7x7, groups, fused pool, padded heads, 4 n-tiles) against
    a plain CPU loop."""
    r = subprocess.run([os.path.join(ROOT, "build", "test_conv_tc")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0 and "ALL OK" in r.stdout


@pytest.mark.parametrize("mode,tol", [("fp32", FP32_TOL), ("bf16x3", BF16X3_TOL), ("bf16", BF16_TOL)])
def test_net_all_stages_vs_oracle_small(native_net, he_sd, mode, tol):
    x = torch.rand((2, 3, 64, 72), generator=torch.Generator().manual_seed(5)) - 0.5
    with torch.no_grad():
        _, saved = net_port.forward(he_sd, x)
    outs = _forward(native_net, x, mode)
    errs = [float((o - s).abs().max()) for o, s in zip(outs, saved)]
    print("mode %s per-stage max|err|: %s" % (mode, " ".join("%.2e" % e for e in errs)))
    assert max(errs) < tol
    assert float(saved[-1].abs().max()) > 0.3


@pytest.mark.parametrize("mode,tol", [("fp32", FP32_TOL), ("bf16x3", BF16X3_TOL), ("bf16", BF16_TOL)])
def test_net_368_vs_reference_golden(native_net, mode, tol):
    g = golden("net_368")
    x = torch.rand((1, 3, 368, 368), generator=torch.Generator().manual_seed(int(g["seed"]))) - 0.5
    outs = _forward(native_net, x, mode)
    e_paf = float(np.abs(outs[10].numpy() - g["paf"]).max())
    e_heat = float(np.abs(outs[11].numpy() - g["heat"]).max())
    print("368x368 %s: max|paf err| %.3e max|heat err| %.3e (|paf|max %.2f)" % (mode, e_paf, e_heat, np.abs(g["paf"]).max()))
    assert e_paf < tol and e_heat < tol
    np.testing.assert_allclose([float(o.abs().max()) for o in outs], g["stage_absmax"], rtol=0.05 if mode == "bf16" else 1e-3)


def test_fp32_mode_is_bit_identical_to_the_exact_oracle(native_net, he_sd):
    """The fp32 mode accumulates every output in the order oracle/conv_exact.c defines (tap-major, cin-minor fused
    multiply-adds from +0, then + bias): all 12 stage outputs must be BIT-identical, not merely within 1e-3."""
    x = torch.rand((2, 3, 64, 72), generator=torch.Generator().manual_seed(5)) - 0.5
    _, saved = net_exact.forward(he_sd, x.numpy())
    outs = _forward(native_net, x, "fp32")
    for i, (o, s_) in enumerate(zip(outs, saved)):
        np.testing.assert_array_equal(o.numpy(), s_, err_msg="stage output %d" % i)


def _oracle_humans(he_sd, frames):
    """The CPU pipeline of the north star: rtpose_preprocess -> exact fp32 network -> NMS -> pafprocess (C port)."""
    port = pafprocess_oracle.load_port()
    x = np.stack([glue_port.rtpose_preprocess(f) for f in frames])
    (paf, heat), _ = net_exact.forward(he_sd, x)
    return [glue_port.paf_to_pose(np.ascontiguousarray(heat[i].transpose(1, 2, 0)),
                                  np.ascontiguousarray(paf[i].transpose(1, 2, 0)), port)[1] for i in range(len(frames))]


def _humans_equal(a, b):
    return (len(a) == len(b) and all(ga[1].keys() == gb[1].keys() and ga[0] == gb[0] and
                                     all(ga[1][k] == gb[1][k] for k in ga[1]) for ga, gb in zip(a, b)))


def test_image_to_humans_identical_keypoint_assignments(built, he_sd):
    """BASELINE.json north_star: "identical keypoint assignments on a fixed synthetic batch".  A fixed seeded batch of
    368x368 uint8 frames goes image -> GPU network (fp32 mode) -> GPU post-processing through the fused engine, and
    through the oracle pipeline on the CPU; persons, parts, coordinates and scores must be identical.  (Random-weight
    maps carry ~4000 peaks per frame and the reference algorithm flips decisions under 3e-5 map perturbations, so this
    only holds because the fp32 mode is bit-identical to the oracle network.)  The tensor-core modes are run on the same
    batch and the number of persons that differ is printed: the price of the fast modes, on record."""
    eng = pkg_module("engine")
    rs = np.random.RandomState(2024)
    frames = rs.randint(0, 256, (4, 368, 368, 3)).astype(np.uint8)
    yy, xx = np.mgrid[0:368, 0:368]
    for i in (2, 3):     # two smooth frames (blobs on a gradient) next to the two noise frames
        img = np.zeros((368, 368, 3), np.float32) + rs.uniform(60, 200, 3)
        for _ in range(10):
            cx, cy, sg = rs.uniform(0, 368), rs.uniform(0, 368), rs.uniform(8, 60)
            img += np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * sg * sg))[:, :, None] * rs.uniform(-120, 120, 3)
        frames[i] = np.clip(img, 0, 255).astype(np.uint8)
    want = _oracle_humans(he_sd, frames)
    arrays = [v.numpy() for v in he_sd.values()]
    pe = eng.PoseEngine(arrays, 0, mode="fp32", batch_cap=4, peak_cap=2048, human_cap=2048)
    got = pe.infer_batch(frames)
    assert sum(len(w) for w in want) > 100
    for i in range(4):
        assert_humans_equal(got[i], want[i], score_tol=0.0)
        assert _humans_equal(got[i], want[i])
    print("fp32 mode: %s persons per frame, all identical to the CPU pipeline" % [len(w) for w in want])
    for mode in ("bf16x3", "bf16"):
        pe_m = eng.PoseEngine(arrays, 0, mode=mode, batch_cap=4, peak_cap=2048, human_cap=2048)
        other = pe_m.infer_batch(frames)
        same_frames = sum(_humans_equal(other[i], want[i]) for i in range(4))
        def keyset(hs):
            return {tuple(sorted((p, round(v[0], 6), round(v[1], 6)) for p, v in h[1].items())) for h in hs}
        common = sum(len(keyset(other[i]) & keyset(want[i])) for i in range(4))
        print("%s mode: persons per frame %s; %d of 4 frames identical; %d of %d reference persons reproduced exactly "
              "(same parts at the same pixels)" % (mode, [len(o) for o in other], same_frames, common,
                                                   sum(len(w) for w in want)))


def test_batch_rows_are_independent_and_deterministic(native_net):
    """Size-independent property at the full bench shape: image i of a batch of 32 equals image i run alone (bit for
    bit), and two runs are identical."""
    x = torch.rand((32, 3, 368, 368), generator=torch.Generator().manual_seed(9)) - 0.5
    a = _forward(native_net, x, "bf16")
    b = _forward(native_net, x, "bf16")
    for i in (10, 11):
        assert torch.equal(a[i], b[i])
    for idx in (0, 17, 31):
        single = _forward(native_net, x[idx:idx + 1], "bf16")
        assert torch.equal(single[10][0], a[10][idx]) and torch.equal(single[11][0], a[11][idx])


def test_module_surface_matches_native(built, he_sd):
    import lib.network.rtpose_vgg as m
    model = m.get_model("vgg19")
    model.load_state_dict(he_sd)
    model = torch.nn.DataParallel(model).cuda()      # demo/picture_demo.py:47
    model.float()
    model.eval()
    x = torch.rand((1, 3, 64, 64), generator=torch.Generator().manual_seed(3)) - 0.5
    model.module.precision = "fp32"
    with torch.no_grad():
        (paf, heat), saved = model(x.cuda())
        (paf_o, heat_o), saved_o = net_port.forward(he_sd, x)
    assert len(saved) == 12 and paf.shape == (1, 38, 8, 8) and heat.shape == (1, 19, 8, 8) and paf.is_cuda
    assert float((paf.cpu() - paf_o).abs().max()) < FP32_TOL and float((heat.cpu() - heat_o).abs().max()) < FP32_TOL
    for s, so in zip(saved, saved_o):
        assert float((s.cpu() - so).abs().max()) < FP32_TOL


@pytest.mark.parametrize("name", sorted(POST_CASES))
def test_post_kernels_vs_oracle_and_reference_golden(name, built):
    eng = pkg_module("engine")
    heat, paf = POST_CASES[name](synth)
    h, w = heat.shape[:2]
    post = eng.NativePost(0, batch_cap=1, peak_cap=1024, human_cap=1024)
    post.run(heat.ctypes.data, paf.ctypes.data, False, 1, 1, h, w, 0.1)
    post.sync()
    post.check_status(1)
    # peaks: identical to the oracle NMS (coordinates, ids, parts AND scores: same float ops in the same order)
    jl = nms_port.joint_list_from_nms(nms_port.nms(heat, 0.1))
    got_jl = post.peaks(0)
    assert got_jl.shape == jl.shape
    np.testing.assert_array_equal(got_jl, jl)
    # humans: identical to the oracle port and to the reference's golden output
    _, want = glue_port.paf_to_pose(heat, paf, pafprocess_oracle.load_port())
    got = eng.humans_to_dicts(post.humans(0), w * 8, h * 8)
    assert_humans_equal(got, want, score_tol=0.0)
    assert_humans_equal(got, humans_rows_to_dicts(golden("post_" + name)["humans"]), score_tol=1e-6)
    print(name, "peaks", len(jl), "humans", len(got), "status", post.status(0))


def test_device_sort_kernels_reproduce_std_sort(built):
    """The product's sorting stages (global-memory partitions above 4096 keys, level-synchronous shared-memory introsort
    below) against the sequential restatement of libstdc++'s std::sort, INCLUDING the order of equal keys, on duplicate-
    heavy and adversarial inputs (sorted / reversed / organ pipe / few distinct values) of every size class."""
    import ctypes
    eng, nat = pkg_module("engine"), pkg_module("_native")
    host = ctypes.CDLL(os.path.join(ROOT, "build", "libpostcore_host.so"))
    U = ctypes.POINTER(ctypes.c_uint64)
    host.core_seq_sort.argtypes = [U, ctypes.c_int, U]
    post = eng.NativePost(0, batch_cap=1, peak_cap=64, human_cap=16)
    rs = np.random.RandomState(0)
    checked = 0

    def check(hi):
        nonlocal checked
        n = len(hi)
        keys = (hi.astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)
        want, got = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        host.core_seq_sort(keys.ctypes.data_as(U), n, want.ctypes.data_as(U))
        nat.check(nat.lib().b200pose_post_debug_sort(post._h, keys.ctypes.data, n, got.ctypes.data), "debug_sort")
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, "n=%d: first mismatch at %d of %d (%d wrong)" % (n, bad[0], n, bad.size)
        checked += 1
    for n in [1, 2, 3, 15, 16, 17, 18, 31, 32, 33, 64, 65, 100, 257, 1000, 2048, 4095, 4096, 4097, 5000, 9000, 20000,
              70000, 300000]:
        for distinct in (1, 2, 7, max(1, n // 3), 1 << 30):
            check(rs.randint(0, distinct, size=n))
    for n in (17, 33, 100, 1000, 4096, 5000, 50000):
        for hi in (np.arange(n), np.arange(n)[::-1], np.minimum(np.arange(n), np.arange(n)[::-1]), np.arange(n) % 2,
                   np.arange(n) % 17, (np.arange(n) * 7919) % 1013):
            check(np.ascontiguousarray(hi))
    print("device std::sort: %d inputs identical to the sequential restatement" % checked)


def test_post_batch_and_nchw_layout(built):
    eng = pkg_module("engine")
    maps = [synth.stick_figures(p, s)[:2] for p, s in ((2, 21), (6, 22), (12, 23), (1, 24))]
    heat = np.stack([m[0] for m in maps]).transpose(0, 3, 1, 2).copy()      # NCHW
    paf = np.stack([m[1] for m in maps]).transpose(0, 3, 1, 2).copy()
    post = eng.NativePost(0, batch_cap=4, peak_cap=256, human_cap=128)
    post.run(heat.ctypes.data, paf.ctypes.data, False, 0, 4, 46, 46, 0.1)
    post.sync()
    post.check_status(4)
    port = pafprocess_oracle.load_port()
    for i, (hm, pf) in enumerate(maps):
        _, want = glue_port.paf_to_pose(hm, pf, port)
        assert_humans_equal(eng.humans_to_dicts(post.humans(i), 368, 368), want, score_tol=0.0)


def test_capacity_overflow_is_loud(built):
    eng, nat = pkg_module("engine"), pkg_module("_native")
    heat, paf = synth.noise_maps(1)
    post = eng.NativePost(0, batch_cap=1, peak_cap=64, human_cap=16)
    post.run(heat.ctypes.data, paf.ctypes.data, False, 1, 1, 46, 46, 0.1)
    post.sync()
    with pytest.raises(nat.B200PoseError):
        post.check_status(1)


def test_legacy_pafprocess_surface(built):
    """lib.pafprocess.pafprocess called exactly like the SWIG module (upsampled maps, getters)."""
    from lib.pafprocess import pafprocess
    port = pafprocess_oracle.load_port()
    for persons, seed in ((3, 3), (8, 8), (30, 30)):
        heat, paf, _ = synth.stick_figures(persons, seed)
        jl = nms_port.joint_list_from_nms(nms_port.nms(heat, 0.1))
        paf_up = np.ascontiguousarray(np.repeat(np.repeat(paf, 8, 0), 8, 1))
        heat_up = np.ascontiguousarray(np.repeat(np.repeat(heat, 8, 0), 8, 1))
        assert pafprocess.process_paf(jl[None], heat_up, paf_up) == 0
        port.process_paf(jl[None], heat_up, paf_up)
        assert pafprocess.get_num_humans() == port.get_num_humans() > 0
        for hid in range(port.get_num_humans()):
            assert pafprocess.get_score(hid) == port.get_score(hid)
            for p in range(18):
                c = pafprocess.get_part_cid(hid, p)
                assert c == port.get_part_cid(hid, p)
                if c >= 0:
                    assert (pafprocess.get_part_x(c), pafprocess.get_part_y(c), pafprocess.get_part_score(c)) == \
                           (port.get_part_x(c), port.get_part_y(c), port.get_part_score(c))
    with pytest.raises(TypeError):
        pafprocess.process_paf(jl[None].astype(np.float64), heat_up, paf_up)


def test_reference_shaped_pipeline_end_to_end(built, he_sd):
    """get_outputs + paf_to_pose_cpp (the calls demo/picture_demo.py makes) vs the oracle glue, fp32 mode."""
    from evaluate.coco_eval import get_outputs
    from lib.config import cfg
    from lib.network.rtpose_vgg import get_model
    from lib.utils.paf_to_pose import NMS, paf_to_pose_cpp
    model = get_model("vgg19")
    model.load_state_dict(he_sd)
    model = model.cuda().float().eval()
    model.precision = "fp32"
    g = golden("get_outputs_200x230")
    img = np.random.RandomState(0).randint(0, 256, (200, 230, 3)).astype(np.uint8)
    with torch.no_grad():
        paf, heat, scale = get_outputs(img, model, "rtpose")
    assert paf.shape == (46, 53, 38) and heat.shape == (46, 53, 19) and abs(scale - float(g["scale"])) < 1e-12
    assert np.abs(paf - g["paf"]).max() < FP32_TOL and np.abs(heat - g["heat"]).max() < FP32_TOL

    # get_outputs took the device path (frame uploaded as bytes, crop_with_factor + normalisation as kernels); the
    # reference's own sequence (host cv2 resize, host normalisation, model(batch)) through the same network must give
    # the very same maps, for every normalisation the reference offers
    class Opaque(torch.nn.Module):          # hides maps_from_frame: get_outputs falls back to the reference sequence
        def __init__(self, inner):
            super().__init__()
            self.inner = inner

        def forward(self, x):
            return self.inner(x)
    for pre in ("rtpose", "vgg", "inception", "ssd"):
        with torch.no_grad():
            a = get_outputs(img, model, pre)
            b = get_outputs(img, Opaque(model), pre)
        np.testing.assert_array_equal(a[0], b[0], err_msg=pre)
        np.testing.assert_array_equal(a[1], b[1], err_msg=pre)
        assert a[2] == b[2]
    # post-processing on the REFERENCE's maps so that the comparison is exact
    humans = paf_to_pose_cpp(g["heat"], g["paf"], cfg)
    _, want = glue_port.paf_to_pose(g["heat"], g["paf"], pafprocess_oracle.load_port())
    got = [(h.score, {p: (b.x, b.y, b.score) for p, b in h.body_parts.items()}) for h in humans]
    assert_humans_equal(got, want, score_tol=0.0)
    per_joint = NMS(g["heat"], upsampFactor=8, config=cfg)
    ref_pj = nms_port.nms(g["heat"], 0.1)
    for a, b in zip(per_joint, ref_pj):
        np.testing.assert_array_equal(a, b.astype(np.float32).astype(np.float64))
    assert paf_to_pose_cpp(np.zeros((46, 46, 19), np.float32), np.zeros((46, 46, 38), np.float32), cfg) == []


def test_fused_engine_matches_stagewise(built, he_sd):
    """b200pose_infer (maps never leave the device) == forward + separate post on the same maps."""
    eng = pkg_module("engine")
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=4, peak_cap=1024, human_cap=1024)
    x = (np.random.RandomState(3).rand(4, 3, 368, 368).astype(np.float32) - 0.5)
    fused = pe.infer_batch(x)
    outs = [torch.empty((4, 38 if i % 2 == 0 else 19, 46, 46), device="cuda") for i in range(12)]
    xd = torch.from_numpy(x).cuda()
    pe.net.forward_ptr(xd.data_ptr(), True, 4, 368, 368, pe.mode, [o.data_ptr() for o in outs], True,
                       torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    port = pafprocess_oracle.load_port()
    for i in range(4):
        heat = outs[11][i].permute(1, 2, 0).contiguous().cpu().numpy()
        paf = outs[10][i].permute(1, 2, 0).contiguous().cpu().numpy()
        _, want = glue_port.paf_to_pose(heat, paf, port)
        assert_humans_equal(fused[i], want, score_tol=0.0)
    assert pkg_module("_native").launch_count() > 0


def test_uint8_input_path_fuses_rtpose_preprocess(native_net, he_sd):
    """b200pose_net_forward_u8 (uint8 HWC BGR frames, preprocessing fused into conv1_1) must give the very same maps as
    rtpose_preprocess on the host + the fp32-input entry point, in both modes, and match the oracle in fp32 mode."""
    nat = pkg_module("_native")
    img = np.random.RandomState(11).randint(0, 256, (2, 64, 72, 3)).astype(np.uint8)
    x = torch.from_numpy(np.stack([glue_port.rtpose_preprocess(i) for i in img]))
    xd = torch.from_numpy(img).cuda()
    for mode in ("bf16", "fp32"):
        ref = _forward(native_net, x, mode)
        outs = [torch.empty((2, 38 if i % 2 == 0 else 19, 8, 9), device="cuda") for i in range(12)]
        native_net.forward_u8_ptr(xd.data_ptr(), True, 2, 64, 72, nat.MODES[mode], [o.data_ptr() for o in outs], True,
                                  torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        for a, b in zip(outs, ref):
            assert torch.equal(a.cpu(), b)
    with torch.no_grad():
        _, saved = net_port.forward(he_sd, x)
    assert max(float((o.cpu() - s).abs().max()) for o, s in zip(outs, saved)) < FP32_TOL


def test_graph_replay_equals_plain_launches(native_net):
    """On a real stream the 52 launches of the forward pass are captured into a CUDA graph per (shape, mode, input
    pointer) and replayed; on the legacy default stream they are launched one by one.  Same bits either way, also after
    the input buffer's contents change, after a shape change in between, and for a second input pointer."""
    nat = pkg_module("_native")
    g = torch.Generator().manual_seed(17)
    side = torch.cuda.Stream()

    def run(xd, stream, mode):
        n, _, H, W = xd.shape
        outs = [torch.empty((n, 38 if i % 2 == 0 else 19, H // 8, W // 8), device="cuda") for i in range(12)]
        native_net.forward_ptr(xd.data_ptr(), True, n, H, W, nat.MODES[mode], [o.data_ptr() for o in outs], True,
                               stream.cuda_stream)
        torch.cuda.synchronize()
        return outs

    for mode in ("bf16", "bf16x3"):
        xa = (torch.rand((2, 3, 64, 72), generator=g) - 0.5).cuda()
        xb = (torch.rand((2, 3, 64, 72), generator=g) - 0.5).cuda()
        xc = (torch.rand((1, 3, 96, 64), generator=g) - 0.5).cuda()
        torch.cuda.synchronize()
        for rep in range(3):
            if rep:
                xa.copy_(torch.rand((2, 3, 64, 72), generator=g) - 0.5)      # same pointer, new frames
                torch.cuda.synchronize()
            for xd in (xa, xc, xb, xa):
                want = run(xd, torch.cuda.default_stream(), mode)
                got = run(xd, side, mode)
                for a, b in zip(got, want):
                    assert torch.equal(a, b)
        assert float(want[-1].abs().max()) > 0.05


def test_two_runs_in_flight_results_are_kept_apart(built):
    """Run i+1 may be submitted before run i is read: results land in parity slots of pinned host memory."""
    eng, nat = pkg_module("engine"), pkg_module("_native")
    port = pafprocess_oracle.load_port()
    maps = [synth.stick_figures(p, s)[:2] for p, s in ((4, 31), (9, 32), (2, 33))]
    post = eng.NativePost(0, batch_cap=1, peak_cap=256, human_cap=128)
    tickets = []
    for hm, pf in maps[:2]:
        post.run(hm.ctypes.data, pf.ctypes.data, False, 1, 1, 46, 46, 0.1)
        tickets.append(post.last_ticket())
    assert tickets == [0, 1]
    for t, (hm, pf) in zip(tickets, maps[:2]):
        post.select(t)
        _, want = glue_port.paf_to_pose(hm, pf, port)
        assert_humans_equal(eng.humans_to_dicts(post.humans(0), 368, 368), want, score_tol=0.0)
    post.run(maps[2][0].ctypes.data, maps[2][1].ctypes.data, False, 1, 1, 46, 46, 0.1)
    with pytest.raises(nat.B200PoseError):
        post.select(0)                      # overwritten: only the last two runs are retained
    post.select(2)
    _, want = glue_port.paf_to_pose(maps[2][0], maps[2][1], port)
    assert_humans_equal(eng.humans_to_dicts(post.humans(0), 368, 368), want, score_tol=0.0)


def test_picture_demo_script_runs(built, tmp_path):
    """demo/picture_demo.py: the reference demo's flow (get_model, DataParallel, get_outputs, paf_to_pose_cpp,
    draw_humans, imwrite) on the B200 path, from the repo root like the reference expects."""
    out = tmp_path / "result.png"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "demo", "picture_demo.py"), "--synthetic-weights", "--precision", "fp32",
                        "--out", str(out)],
                       cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0 and out.exists() and "humans" in r.stdout


def test_data_parallel_over_every_visible_gpu(built, he_sd):
    """demo/picture_demo.py:47 wraps the model in DataParallel; with more than one visible GPU torch replicates the
    module (replicas own no parameters) and scatters the batch.  Every replica must find the master's weights and its
    own device's native net; the gathered result equals the single-device run bit for bit."""
    import lib.network.rtpose_vgg as m
    ngpu = torch.cuda.device_count()
    model = m.get_model("vgg19")
    model.load_state_dict(he_sd)
    model.precision = "fp32"
    single = model.cuda().float().eval()
    x = (torch.rand((max(2, ngpu), 3, 64, 64), generator=torch.Generator().manual_seed(3)) - 0.5).cuda()
    with torch.no_grad():
        (paf1, heat1), _ = single(x)
        dp = torch.nn.DataParallel(single)
        (paf2, heat2), saved = dp(x)
    assert len(saved) == 12 and paf2.shape == paf1.shape
    assert torch.equal(paf1.cpu(), paf2.cpu()) and torch.equal(heat1.cpu(), heat2.cpu())
    print("DataParallel over %d GPU(s): identical to the single-device forward" % ngpu)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_sharded_batch_equals_single_gpu(built, he_sd, tmp_path):
    """SURVEY.md 4 / 8(e): a batch sharded over two ranks (one process per GPU, NCCL weight broadcast, shard_range)
    gives, frame by frame, bit-identical persons to the same batch on one GPU."""
    worker = os.path.join(ROOT, "tests", "mgpu_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29713", worker, str(tmp_path)],
                       cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0
    eng = pkg_module("engine")
    frames = np.random.RandomState(77).randint(0, 256, (64, 184, 184, 3)).astype(np.uint8)
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=32, peak_cap=1024, human_cap=1024)
    want = []
    for lo in (0, 32):
        pe.infer_batch(frames[lo:lo + 32])
        want += [a.copy() for a in pe.fetch_arrays()]
    got = [None] * 64
    for rank in (0, 1):
        z = np.load(os.path.join(str(tmp_path), "rank%d.npz" % rank))
        for k in z.files:
            got[int(k)] = z[k]
    assert all(g is not None for g in got)
    for i in range(64):
        np.testing.assert_array_equal(got[i], want[i], err_msg="frame %d" % i)
    print("64 frames over 2 ranks: per-frame persons bit-identical to the 1-GPU run (%d persons)" % sum(len(w) for w in want))
