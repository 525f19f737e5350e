"""GPU (-m gpu): the widened rows of SURVEY.md 8(f) - device-side crop_with_factor (rank 1) and flip test-time
averaging (8(a) F1 / rank 2) - against the oracle (cv2-based crop_with_factor, handle_paf_and_heat), the reference's
golden vectors and the reference-shaped composition
get_outputs(img) + get_outputs(img[:, ::-1]) + handle_paf_and_heat + paf_to_pose."""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, RecordedPafprocess, assert_humans_equal, golden, pkg_module
from oracle import glue_port, pafprocess_oracle, synth

pytestmark = pytest.mark.gpu


def test_flip_harness_through_the_c_abi(built):
    """tests/cuda/test_flip.cpp: fused b200pose_infer*_flip == forward x2 + host merge + post_run, bit for bit, in all
    three arithmetic modes; merge kernel == host core in both layouts; crop_with_factor kernel == host core;
    b200pose_infer_raw_u8 (with and without flip) == host crop + the uint8 entry points."""
    r = subprocess.run([os.path.join(ROOT, "build", "test_flip"), "184", "248", "no-multiscale"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0 and "FLIP TEST OK" in r.stdout, r.stdout[-2000:]


def test_multiscale_harness_through_the_c_abi(built):
    """Same harness including the multi-scale sections: b200pose_infer_raw_u8_multiscale (flip 0 / 1) == per scale host
    crop + validated forward + host merge + host bicubic resize (shared core) + float32 average + validated post_run."""
    r = subprocess.run([os.path.join(ROOT, "build", "test_flip"), "184", "248"], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0 and "FLIP TEST OK" in r.stdout and "multiscale(flip=1)" in r.stdout, r.stdout[-2000:]


def test_flip_merge_kernel_matches_reference_golden(built):
    eng = pkg_module("engine")
    post = eng.NativePost(0, batch_cap=1, peak_cap=64, human_cap=64)
    nh, fh, npf, fpf = [np.random.RandomState(sd).rand(6, 5, c).astype(np.float32)
                        for sd, c in ((1, 19), (2, 19), (3, 38), (4, 38))]
    keep = fpf.copy()
    ap, ah = post.flip_merge(nh, fh, npf, fpf)
    f = golden("flip_merge")                   # produced by the reference's handle_paf_and_heat
    np.testing.assert_array_equal(ap, f["avg_paf"])
    np.testing.assert_array_equal(ah, f["avg_heat"])
    np.testing.assert_array_equal(fpf, keep)   # documented deviation: inputs are not modified in place
    # batch, both layouts, signed values
    rs = np.random.RandomState(9)
    bnh, bfh, bnp, bfp = (rs.randn(3, 46, 53, c).astype(np.float32) for c in (19, 19, 38, 38))
    ap, ah = post.flip_merge(bnh, bfh, bnp, bfp)
    t = lambda a: np.ascontiguousarray(a.transpose(0, 3, 1, 2))
    ap0, ah0 = post.flip_merge(t(bnh), t(bfh), t(bnp), t(bfp), layout=0)
    for i in range(3):
        wp, wh = glue_port.handle_paf_and_heat(bnh[i], bfh[i], bnp[i], bfp[i])
        np.testing.assert_array_equal(ap[i], wp)
        np.testing.assert_array_equal(ah[i], wh)
        np.testing.assert_array_equal(ap0[i], wp.transpose(2, 0, 1))
        np.testing.assert_array_equal(ah0[i], wh.transpose(2, 0, 1))


def test_fused_flip_inference_matches_reference_shaped_composition(built, he_sd):
    """PoseEngine.infer_batch(flip=True) on uint8 frames == per image: forward(img), forward(img[:, ::-1]) (fp32 parity
    mode through the native net), the oracle's handle_paf_and_heat and paf_to_pose on the averaged maps."""
    eng = pkg_module("engine")
    nat = pkg_module("_native")
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=2, peak_cap=1024, human_cap=2048)
    frames = np.random.RandomState(21).randint(0, 256, (2, 184, 248, 3)).astype(np.uint8)
    fused = pe.infer_batch(frames, flip=True)
    both = np.ascontiguousarray(np.concatenate([frames, frames[:, :, ::-1]], 0))
    outs = [torch.empty((4, 38 if i % 2 == 0 else 19, 23, 31), device="cuda") for i in range(12)]
    xd = torch.from_numpy(both).cuda()
    pe.net.forward_u8_ptr(xd.data_ptr(), True, 4, 184, 248, pe.mode, [o.data_ptr() for o in outs], True,
                          torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    paf = outs[10].permute(0, 2, 3, 1).contiguous().cpu().numpy()
    heat = outs[11].permute(0, 2, 3, 1).contiguous().cpu().numpy()
    port = pafprocess_oracle.load_port()
    total = 0
    for i in range(2):
        ap, ah = glue_port.handle_paf_and_heat(heat[i], heat[2 + i], paf[i], paf[2 + i])
        _, want = glue_port.paf_to_pose(ah, ap, port)
        assert_humans_equal(fused[i], want, score_tol=0.0)
        total += len(want)
    plain = pe.infer_batch(frames)
    assert total > 0 and any(len(a) != len(b) or a != b for a, b in zip(plain, fused))   # averaging changed something
    assert nat.launch_count() > 0


def test_pafprocess_kernels_fuzz_against_the_compiled_reference(built):
    """The limbs / assembly kernels (through the legacy lib.pafprocess surface: joint list + x8 maps, exactly what the
    SWIG module gets) on 80 random inputs the fixtures do not reach - duplicated peaks on one pixel, exact score ties,
    cross links between persons, masked fields - against what the reference's own pafprocess.cpp returned on them
    (golden).  Same scenarios as the host-side fuzz in tests/test_host.py."""
    from lib.pafprocess import pafprocess
    ref = RecordedPafprocess()
    humans = 0
    for t in range(80):
        h, w, jl, paf = synth.fuzz_scenario(t)
        if len(jl) == 0:
            continue
        paf_up = np.ascontiguousarray(np.repeat(np.repeat(paf, 8, 0), 8, 1))
        heat_up = np.zeros((h * 8, w * 8, 19), np.float32)
        assert pafprocess.process_paf(jl[None], heat_up, paf_up) == 0
        ref.select(t, jl, paf)
        assert pafprocess.get_num_humans() == ref.get_num_humans(), "scenario seed %d" % (1000 + t)
        for hid in range(ref.get_num_humans()):
            assert pafprocess.get_score(hid) == ref.get_score(hid), "scenario seed %d" % (1000 + t)
            for p in range(18):
                assert pafprocess.get_part_cid(hid, p) == ref.get_part_cid(hid, p), "scenario seed %d" % (1000 + t)
        humans += ref.get_num_humans()
    assert humans > 80


def test_crop_with_factor_kernel_matches_reference_golden_and_cv2(built, he_sd):
    eng = pkg_module("engine")
    net = eng.NativeNet(0)                      # crop_with_factor needs no weights
    f = golden("crop_with_factor")              # produced by the reference's crop_with_factor
    for name, h, w, dest, seed in (("50x61", 50, 61, 96, 5), ("64x71_half", 64, 71, 32, 6), ("30x22_up", 30, 22, 40, 7)):
        img = np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)
        out, scale, shape = net.crop_with_factor(img, dest, 8)
        np.testing.assert_array_equal(out, f[name + "_out"])
        assert [scale, shape[0], shape[1]] == list(f[name + "_meta"])
    rs = np.random.RandomState(4)
    for (h, w, dest) in ((200, 230, 368), (480, 640, 368), (736, 739, 368), (1080, 1920, 368), (97, 64, 200), (368, 368, 368)):
        frames = rs.randint(0, 256, (2, h, w, 3)).astype(np.uint8)
        out, scale, shape = net.crop_with_factor(frames, dest, 8)
        for i in range(2):
            want, ws, wshape = glue_port.crop_with_factor(frames[i], dest, 8)       # cv2.resize on the host
            assert scale == ws and shape == tuple(wshape)
            np.testing.assert_array_equal(out[i], want)


def test_raw_frames_of_mixed_sizes_match_reference_shaped_pipeline(built, he_sd):
    """PoseEngine.infer_images (device crop_with_factor + net + post, frames bucketed by shape) == per image: the
    oracle's crop_with_factor (cv2), the native uint8 forward, the oracle's paf_to_pose."""
    eng = pkg_module("engine")
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=2, peak_cap=1024, human_cap=2048)
    rs = np.random.RandomState(31)
    imgs = [rs.randint(0, 256, s).astype(np.uint8) for s in ((150, 211, 3), (120, 100, 3), (150, 211, 3))]
    got = pe.infer_images(imgs, dest_size=184, factor=8)
    port = pafprocess_oracle.load_port()
    total = 0
    for i, im in enumerate(imgs):
        crop, _, _ = glue_port.crop_with_factor(im, 184, 8)
        H, W = crop.shape[:2]
        outs = [torch.empty((1, 38 if k % 2 == 0 else 19, H // 8, W // 8), device="cuda") for k in range(12)]
        xd = torch.from_numpy(np.ascontiguousarray(crop[None])).cuda()
        pe.net.forward_u8_ptr(xd.data_ptr(), True, 1, H, W, pe.mode, [o.data_ptr() for o in outs], True,
                              torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        heat = outs[11][0].permute(1, 2, 0).contiguous().cpu().numpy()
        paf = outs[10][0].permute(1, 2, 0).contiguous().cpu().numpy()
        _, want = glue_port.paf_to_pose(heat, paf, port)
        assert_humans_equal(got[i], want, score_tol=0.0)
        total += len(want)
    assert total > 0


def test_multiscale_flip_averaging_matches_composed_oracle(built, he_sd):
    """BASELINE.json configs[4] (multi-scale 0.5/1.0/1.5/2.0 with L/R flip): PoseEngine.infer_images(scales=..., flip=True)
    == per scale the oracle's crop_with_factor of the frame and of the mirrored frame, the native uint8 forward, then the
    oracle's handle_paf_and_heat, bicubic resize to the base grid, float32 average and paf_to_pose."""
    eng = pkg_module("engine")
    pe = eng.PoseEngine([v.numpy() for v in he_sd.values()], 0, mode="bf16", batch_cap=2, peak_cap=1024, human_cap=2048)
    rs = np.random.RandomState(41)
    imgs = [rs.randint(0, 256, (90, 123, 3)).astype(np.uint8) for _ in range(2)]
    scales, base = (0.5, 1.0, 1.5, 2.0), 96
    got = pe.infer_images(imgs, dest_size=base, factor=8, flip=True, scales=scales)
    port = pafprocess_oracle.load_port()

    def maps(frame, dest):
        crop, _, _ = glue_port.crop_with_factor(frame, dest, 8)
        H, W = crop.shape[:2]
        outs = [torch.empty((1, 38 if k % 2 == 0 else 19, H // 8, W // 8), device="cuda") for k in range(12)]
        xd = torch.from_numpy(np.ascontiguousarray(crop[None])).cuda()
        pe.net.forward_u8_ptr(xd.data_ptr(), True, 1, H, W, pe.mode, [o.data_ptr() for o in outs], True,
                              torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return (outs[11][0].permute(1, 2, 0).contiguous().cpu().numpy(), outs[10][0].permute(1, 2, 0).contiguous().cpu().numpy())
    total = 0
    for i, im in enumerate(imgs):
        base_crop, _, _ = glue_port.crop_with_factor(im, base, 8)
        per_scale = []
        for s in scales:
            heat, paf = maps(im, int(base * s))
            heat_f, paf_f = maps(np.ascontiguousarray(im[:, ::-1]), int(base * s))
            per_scale.append((heat, paf, heat_f, paf_f))
        ah, ap = glue_port.multi_scale_maps(per_scale, (base_crop.shape[0] // 8, base_crop.shape[1] // 8))
        _, want = glue_port.paf_to_pose(ah, ap, port)
        assert_humans_equal(got[i], want, score_tol=0.0)
        total += len(want)
    assert total > 0


def test_every_preprocess_mode_fused_into_conv1_1(built, he_sd):
    """b200pose_net_set_preprocess: the uint8 entry point with 'vgg' / 'inception' / 'ssd' / 'rtpose' fused into the first
    convolution gives the very same maps as the numpy function on the host + the fp32-input entry point (bf16 and fp32
    modes)."""
    eng = pkg_module("engine")
    nat = pkg_module("_native")
    pre = pkg_module("lib.datasets.preprocessing")
    net = eng.NativeNet(0)
    net.load_state_dict_arrays([v.numpy() for v in he_sd.values()])
    img = np.random.RandomState(17).randint(0, 256, (2, 64, 72, 3)).astype(np.uint8)
    xd = torch.from_numpy(img).cuda()
    stream = torch.cuda.current_stream().cuda_stream
    for name, fn in (("vgg", pre.vgg_preprocess), ("inception", pre.inception_preprocess), ("ssd", pre.ssd_preprocess),
                     ("rtpose", pre.rtpose_preprocess)):
        net.set_preprocess(name)
        xf = torch.from_numpy(np.stack([fn(i) for i in img])).cuda().contiguous()
        for mode in ("bf16", "fp32"):
            a = [torch.empty((2, 38 if i % 2 == 0 else 19, 8, 9), device="cuda") for i in range(12)]
            b = [torch.empty_like(t) for t in a]
            net.forward_u8_ptr(xd.data_ptr(), True, 2, 64, 72, nat.MODES[mode], [o.data_ptr() for o in a], True, stream)
            net.forward_ptr(xf.data_ptr(), True, 2, 64, 72, nat.MODES[mode], [o.data_ptr() for o in b], True, stream)
            torch.cuda.synchronize()
            for u, v in zip(a, b):
                assert torch.equal(u, v), (name, mode)
    with pytest.raises(nat.B200PoseError):
        net.set_preprocess("caffe")
