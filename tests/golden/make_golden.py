"""Generates the committed golden fixtures by running the UNMODIFIED reference (/root/reference) in this
container (it cannot travel to the GPU box).  Usage:  python tests/golden/make_golden.py

Shims needed to import the reference here (none of them touches its arithmetic):
  * stub modules for yacs / pycocotools / matplotlib / pylab (absent offline),
  * lib.pafprocess.pafprocess = ctypes view of oracle/_ref/libpafprocess_ref.so (the reference's own
    pafprocess.cpp compiled as-is; SWIG is absent),
  * torch.Tensor.cuda patched to identity for get_outputs (hard-coded .cuda(), coco_eval.py:108).
Inputs are regenerated from seeds by oracle/synth.py and oracle/net_port.he_state_dict; each fixture stores a
checksum of its inputs so drift is detected.
"""
import hashlib
import os
import sys
import types

ARGS = sys.argv[1:]     # optional: "crop" / "eval" / "pre" / "paf" / "scripts" regenerate only those small fixtures

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from oracle import net_port, pafprocess_oracle, synth  # noqa: E402


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def import_reference():
    import yaml

    class CN(dict):
        def __init__(self, init=None, new_allowed=False):
            super().__init__(init or {})
        __getattr__ = dict.__getitem__
        __setattr__ = dict.__setitem__

        def defrost(self): pass
        def freeze(self): pass

        def merge_from_file(self, f):
            def rec(dst, src):
                for k, v in src.items():
                    if isinstance(v, dict):
                        dst.setdefault(k, CN())
                        rec(dst[k], v)
                    else:
                        dst[k] = v
            rec(self, yaml.safe_load(open(f)))

        def merge_from_list(self, l): pass

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    stub("yacs"); stub("yacs.config", CfgNode=CN)
    stub("pycocotools"); stub("pycocotools.coco", COCO=object); stub("pycocotools.cocoeval", COCOeval=object)
    stub("matplotlib"); stub("matplotlib.pyplot"); stub("pylab")
    for k in [k for k in sys.modules if k == "lib" or k.startswith("lib.") or k == "evaluate" or k.startswith("evaluate.")]:
        del sys.modules[k]
    sys.path.insert(0, REF)
    pafprocess_oracle.build(ref=True)
    ref_paf = pafprocess_oracle.load_ref()
    import lib.pafprocess as lp   # the reference's package (empty __init__)
    mod = types.ModuleType("lib.pafprocess.pafprocess")
    for n in ("process_paf", "get_num_humans", "get_part_cid", "get_score", "get_part_x", "get_part_y", "get_part_score"):
        setattr(mod, n, getattr(ref_paf, n))
    sys.modules["lib.pafprocess.pafprocess"] = mod
    lp.pafprocess = mod
    from lib.network.rtpose_vgg import get_model
    from lib.utils import paf_to_pose as ref_p2p
    sys.argv = ["x", "--cfg", os.path.join(REF, "experiments/vgg19_368x368_sgd.yaml")]
    from evaluate import coco_eval as ref_eval
    from lib.config import cfg
    return get_model, ref_p2p, ref_eval, cfg


CROP_CASES = (("50x61", 50, 61, 96, 5), ("64x71_half", 64, 71, 32, 6), ("30x22_up", 30, 22, 40, 7))


def make_crop():
    """crop_with_factor (lib/network/im_transform.py:119-134) of the reference on seeded uint8 frames: general bilinear
    down-scaling, an exact 2x reduction with a cut last column (cv2 switches to INTER_AREA), up-scaling."""
    from lib.network import im_transform as ref_tf
    out = {}
    for name, h, w, dest, seed in CROP_CASES:
        img = np.random.RandomState(seed).randint(0, 256, (h, w, 3)).astype(np.uint8)
        croped, scale, shape = ref_tf.crop_with_factor(img, dest, factor=8, is_ceil=True)
        out[name + "_out"] = croped
        out[name + "_meta"] = np.array([scale, shape[0], shape[1]], np.float64)
        out[name + "_digest"] = digest(img)
        print("crop", name, img.shape, "->", shape, croped.shape, scale)
    np.savez_compressed(os.path.join(OUT, "crop_with_factor.npz"), **out)


def eval_humans(Human, BodyPart, seed=17, count=5):
    """Seeded synthetic persons (some parts missing) for the append_result fixture; the same generator is used by the
    test with the product's Human / BodyPart classes."""
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


def make_eval(ref_eval):
    """append_result (evaluate/coco_eval.py:117-154) of the reference on seeded persons."""
    from lib.utils.common import BodyPart, Human
    outputs = []
    ref_eval.append_result(42, eval_humans(Human, BodyPart), (368 / 0.71, 496 / 0.71), outputs)
    np.savez_compressed(os.path.join(OUT, "append_result.npz"),
                        keypoints=np.array([o["keypoints"] for o in outputs], np.float64),
                        score=np.array([o["score"] for o in outputs], np.float64),
                        image_id=np.array([o["image_id"] for o in outputs]),
                        category_id=np.array([o["category_id"] for o in outputs]),
                        keys=np.array(list(outputs[0].keys())))
    print("append_result", len(outputs), "records")


def make_preprocess():
    """The four image normalisations of the reference (lib/datasets/preprocessing.py) on an image that holds every
    uint8 value in every channel."""
    from lib.datasets import preprocessing as ref_pre
    img = np.zeros((16, 16, 3), np.uint8)
    img[:, :, 0] = np.arange(256).reshape(16, 16)
    img[:, :, 1] = np.arange(256)[::-1].reshape(16, 16)
    img[:, :, 2] = (np.arange(256) * 7 % 256).reshape(16, 16)
    np.savez_compressed(os.path.join(OUT, "preprocess.npz"), img=img, rtpose=ref_pre.rtpose_preprocess(img.copy()),
                        vgg=ref_pre.vgg_preprocess(img.copy()), inception=ref_pre.inception_preprocess(img.copy()),
                        ssd=ref_pre.ssd_preprocess(img.copy()))
    print("preprocess fixture written")


def post_cases():
    return [("p1", synth.stick_figures(1, 1)[:2]), ("p3", synth.stick_figures(3, 3)[:2]),
            ("p8", synth.stick_figures(8, 8)[:2]), ("p30", synth.stick_figures(30, 30)[:2]),
            ("noise0", synth.noise_maps(0)), ("empty", (np.zeros((46, 46, 19), np.float32), np.zeros((46, 46, 38), np.float32))),
            ("p5_40x52", synth.stick_figures(5, 55, h=40, w=52)[:2])]


FUZZ_SCENARIOS = 300
TIES_CASES = ((30, 31), (50, 5), (80, 7))


def make_pafprocess():
    """The reference's own pafprocess.cpp (oracle/_ref, compiled as-is) on the inputs the tests feed it:
      * fuzz_*: the getters after process_paf on synth.fuzz_scenario(t), t < FUZZ_SCENARIOS (heat_up all zero, paf
        upsampled x8 by repetition); fuzz_humans[t] = -1 marks a scenario without peaks (never run);
      * post_<case> / ties_<persons>_<seed>: glue_port.paf_to_pose (the oracle's NMS, then the reference's pafprocess)
        as humans rows [k, 1 + 18 * 3] in float64, exact."""
    from oracle import glue_port
    pafprocess_oracle.build(ref=True)
    ref = pafprocess_oracle.load_ref()
    digests, counts, scores, cids, parts = [], [], [], [], []
    for t in range(FUZZ_SCENARIOS):
        h, w, jl, paf = synth.fuzz_scenario(t)
        digests.append(digest(jl, paf))
        if len(jl) == 0:
            counts.append(-1)
            continue
        paf_up = np.ascontiguousarray(np.repeat(np.repeat(paf, 8, axis=0), 8, axis=1))
        ref.process_paf(jl[None], np.zeros((h * 8, w * 8, 19), np.float32), paf_up)
        counts.append(ref.get_num_humans())
        for hid in range(ref.get_num_humans()):
            scores.append(ref.get_score(hid))
            c = [int(ref.get_part_cid(hid, p)) for p in range(18)]
            cids.append(c)
            parts.append([(ref.get_part_x(k), ref.get_part_y(k), ref.get_part_score(k)) if k >= 0 else (-1, -1, -1)
                          for k in c])
    out = dict(fuzz_digest=np.array(digests), fuzz_humans=np.array(counts, np.int32),
               fuzz_score=np.array(scores, np.float32), fuzz_cid=np.array(cids, np.int32).reshape(-1, 18),
               fuzz_part=np.array(parts, np.float64).reshape(-1, 18, 3))

    def rows(humans):
        r = np.full((len(humans), 1 + 18 * 3), -1.0, np.float64)
        for i, (score, body) in enumerate(humans):
            r[i, 0] = score
            for p, v in body.items():
                r[i, 1 + 3 * p: 4 + 3 * p] = v
        return r
    for name, (heat, paf) in post_cases():
        out["post_" + name] = rows(glue_port.paf_to_pose(heat, paf, ref)[1])
    for persons, seed in TIES_CASES:
        heat, paf, _ = synth.stick_figures(persons, seed)
        out["ties_%d_%d" % (persons, seed)] = rows(glue_port.paf_to_pose(heat, paf, ref)[1])
    np.savez_compressed(os.path.join(OUT, "pafprocess_ref.npz"), **out)
    print("pafprocess: %d fuzz scenarios, %d humans" % (FUZZ_SCENARIOS, len(scores)))


def make_scripts():
    """The reference's demo/picture_demo.py and evaluate/evaluation.py executed unmodified from this repository's root
    up to their first .cuda(), as tests/test_reference_scripts.py does: the record of each run.  Runs in a process of
    its own, with this repository's lib.* / evaluate.* (import_reference() puts the reference's in their place)."""
    import json
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_reference_scripts
    sd = net_port.he_state_dict(1234)
    ckpt = {"state_dict": {"model." + k: v for k, v in sd.items()}}
    out = {}
    for rel, ckpt_of in (("demo/picture_demo.py", sd), ("evaluate/evaluation.py", ckpt)):
        out[rel] = test_reference_scripts.run_reference_script(os.path.join(REF, rel), lambda *a, **k: ckpt_of)[1]
        print(rel, "reaches .cuda() on", out[rel]["cuda_on"], "after", len(out[rel]["imports"]), "imports")
    with open(os.path.join(OUT, "reference_scripts.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


def main():
    import torch
    if ARGS == ["scripts"]:
        make_scripts()
        return
    if not ARGS or "scripts" in ARGS:
        import subprocess
        subprocess.run([sys.executable, os.path.abspath(__file__), "scripts"], check=True)
    if not ARGS or "paf" in ARGS:
        make_pafprocess()           # needs only the compiled pafprocess.cpp
    if ARGS and set(ARGS) <= {"paf", "scripts"}:
        return
    get_model, ref_p2p, ref_eval, cfg = import_reference()
    if not ARGS or "pre" in ARGS:
        make_preprocess()
    if not ARGS or "crop" in ARGS:
        make_crop()
    if not ARGS or "eval" in ARGS:
        make_eval(ref_eval)
    if ARGS and set(ARGS) <= {"crop", "eval", "pre", "paf", "scripts"}:
        return
    torch.manual_seed(0)

    # ---------------- network (rtpose_model.forward) ----------------
    sd = net_port.he_state_dict(1234)
    model = get_model('vgg19')
    model.load_state_dict(sd, strict=True)
    model.eval()
    for name, hw, seed in (("net_64", 64, 11), ("net_368", 368, 1234)):
        g = torch.Generator().manual_seed(seed)
        x = torch.rand((1, 3, hw, hw), generator=g) - 0.5
        with torch.no_grad():
            (paf, heat), saved = model(x)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), seed=seed, hw=hw, x_digest=digest(x.numpy()),
                            paf=paf.numpy(), heat=heat.numpy(),
                            stage_absmax=np.array([float(t.abs().max()) for t in saved]),
                            stage_mean=np.array([float(t.double().mean()) for t in saved]),
                            stage_sample=np.stack([t.numpy().reshape(-1)[::13][:64] for t in saved]))
        print(name, "paf absmax %.3f heat absmax %.3f" % (paf.abs().max(), heat.abs().max()))

    # ---------------- get_outputs glue on a synthetic uint8 image (non-square: exercises crop_with_factor) -----
    img = np.random.RandomState(0).randint(0, 256, (200, 230, 3)).astype(np.uint8)
    torch.Tensor.cuda = lambda self, *a, **k: self
    with torch.no_grad():
        paf, heat, scale = ref_eval.get_outputs(img, model, 'rtpose')
    np.savez_compressed(os.path.join(OUT, "get_outputs_200x230.npz"), img_digest=digest(img), paf=paf, heat=heat,
                        scale=scale)
    print("get_outputs", paf.shape, heat.shape, scale)
    nh, fh = np.random.RandomState(1).rand(6, 5, 19).astype(np.float32), np.random.RandomState(2).rand(6, 5, 19).astype(np.float32)
    npf, fpf = np.random.RandomState(3).rand(6, 5, 38).astype(np.float32), np.random.RandomState(4).rand(6, 5, 38).astype(np.float32)
    ap, ah = ref_eval.handle_paf_and_heat(nh.copy(), fh.copy(), npf.copy(), fpf.copy())
    np.savez_compressed(os.path.join(OUT, "flip_merge.npz"), avg_paf=ap, avg_heat=ah)

    # ---------------- post-processing (NMS + paf_to_pose_cpp with the compiled pafprocess.cpp) ----------------
    for name, (heat, paf) in post_cases():
        per_joint = ref_p2p.NMS(heat, upsampFactor=cfg.MODEL.DOWNSAMPLE, config=cfg)
        jl = np.array([tuple(p) + (j,) for j, peaks in enumerate(per_joint) for p in peaks]).astype(np.float32).reshape(-1, 5)
        humans = ref_p2p.paf_to_pose_cpp(heat, paf, cfg)
        rows = np.full((len(humans), 1 + 18 * 3), -1.0, np.float64)
        for i, hm in enumerate(humans):
            rows[i, 0] = hm.score
            for p, bp in hm.body_parts.items():
                rows[i, 1 + 3 * p: 4 + 3 * p] = (bp.x, bp.y, bp.score)
        np.savez_compressed(os.path.join(OUT, "post_%s.npz" % name), in_digest=digest(heat, paf), joint_list=jl,
                            humans=rows, shape=np.array(heat.shape[:2]))
        print(name, "peaks", len(jl), "humans", len(humans))


if __name__ == "__main__":
    main()
