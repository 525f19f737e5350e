"""BASELINE.json north_star: "... so evaluate/evaluation.py and demo/picture_demo.py run unmodified".

CPU part: the reference's OWN two scripts, executed unmodified from this repository's root against its `lib.*` /
`evaluate.*` modules, up to their first `.cuda()` - the point where a GPU becomes necessary.  Third-party modules the
scripts import but never use on this path (`pylab`, `matplotlib`) are stubbed and `torch.load` hands out a synthetic
checkpoint.  What such a run does is recorded in tests/golden/reference_scripts.json (tests/golden/make_golden.py
scripts): the imports each script makes from `lib.*` / `evaluate.*`, its parsed command line and the class of the module
`.cuda()` is called on.  The tests make those imports again from this repository and run the calls before `.cuda()`
(argparse values + update_config on the shipped yaml, get_model, load_state_dict with the reference's key names,
DataParallel), and check that the calls after it bind.  With a checkout of the reference named by
B200POSE_REFERENCE_DIR they also execute the scripts themselves and check that the run still matches the record.
Nothing of the scripts is copied.

GPU part: this repo's demo with the reference's command line (no extra flags), on the shipped 674x712 stand-in for
./readme/ski.jpg and a pose_model.pth written by the test."""
import argparse
import builtins
import inspect
import json
import os
import subprocess
import sys
import types

import pytest
import torch

from conftest import GOLDEN, ROOT

REF = os.environ.get("B200POSE_REFERENCE_DIR", "")


class _ReachedCuda(Exception):
    pass


def run_reference_script(path, fake_load):
    """Executes a script of the reference, unmodified, from this repository's root up to its first `.cuda()`.
    Returns its namespace and the record of the run (see the module docstring)."""
    src = open(path).read()
    glob = {"__name__": "__main__", "__file__": path}
    imports = []
    real_import = builtins.__import__

    def import_(name, globals=None, locals=None, fromlist=(), level=0):
        if globals is glob and level == 0 and name.split(".")[0] in ("lib", "evaluate"):
            imports.append([name, list(fromlist or ())])
        return real_import(name, globals, locals, fromlist, level)

    def cuda(self, *a, **k):
        raise _ReachedCuda(type(self).__name__)
    with pytest.MonkeyPatch.context() as mp:
        mp.chdir(ROOT)
        mp.setattr(sys, "argv", [os.path.basename(path)])
        for name in ("pylab", "matplotlib"):
            try:
                __import__(name)
            except ImportError:
                mp.setitem(sys.modules, name, types.ModuleType(name))
        mp.setattr(torch, "load", fake_load)
        mp.setattr(torch.nn.Module, "cuda", cuda)
        mp.setattr(builtins, "__import__", import_)
        with pytest.raises(_ReachedCuda) as ei:
            exec(compile(src, path, "exec"), glob)
    args = glob.get("args")
    return glob, {"imports": imports, "cuda_on": str(ei.value), "args": vars(args) if args is not None else None}


def _recorded(rel, fake_load):
    """The record of script `rel`; checked against a live run when a checkout of the reference is at hand."""
    with open(os.path.join(GOLDEN, "reference_scripts.json")) as f:
        rec = json.load(f)[rel]
    if REF:
        assert run_reference_script(os.path.join(REF, rel), fake_load)[1] == rec, "the record of %s is stale" % rel
    return rec


def _import_as_recorded(rec):
    """The recorded imports, made again from this repository's root: the names they bind in the script."""
    ns = {}
    for module, names in rec["imports"]:
        mod = __import__(module, fromlist=names)        # `from module import names` / `import module`
        for n in names:
            ns[n] = getattr(mod, n)
        if not names:
            ns[module.split(".")[0]] = mod
    return ns


def test_reference_picture_demo_runs_unmodified_up_to_cuda(monkeypatch, built, he_sd):
    rec = _recorded("demo/picture_demo.py", lambda *a, **k: he_sd)
    assert rec["cuda_on"] == "DataParallel"            # model = torch.nn.DataParallel(model).cuda()   (:47)
    monkeypatch.chdir(ROOT)
    glob = _import_as_recorded(rec)
    glob["args"] = argparse.Namespace(**rec["args"])
    glob["update_config"](glob["cfg"], glob["args"])                       # (:44)
    model = glob["get_model"]("vgg19")                                     # (:46-47)
    model.load_state_dict(he_sd)
    torch.nn.DataParallel(model)
    assert len(model.state_dict()) == 184 and torch.equal(model.state_dict()["model0.0.weight"], he_sd["model0.0.weight"])
    assert glob["cfg"].DATASET.IMAGE_SIZE == 368 and glob["args"].weight == "pose_model.pth"
    assert os.path.exists(os.path.join(ROOT, "readme", "ski.jpg"))        # test_image = './readme/ski.jpg'   (:51)
    # the calls the script makes after .cuda() bind to this repo's functions (:58-64)
    inspect.signature(glob["get_outputs"]).bind("oriImg", "model", "rtpose")
    inspect.signature(glob["paf_to_pose_cpp"]).bind("heatmap", "paf", glob["cfg"])
    inspect.signature(glob["draw_humans"]).bind("oriImg", [])
    inspect.signature(glob["handle_paf_and_heat"]).bind(1, 2, 3, 4)
    for name in ("Human", "BodyPart", "CocoPart", "CocoColors", "CocoPairsRender", "im_transform", "update_config"):
        assert name in glob


def test_reference_evaluation_script_runs_unmodified_up_to_cuda(monkeypatch, built, he_sd):
    ckpt = {"state_dict": {"model." + k: v for k, v in he_sd.items()}}     # evaluation.py:15-20 strips 6 characters
    rec = _recorded("evaluate/evaluation.py", lambda *a, **k: ckpt)
    assert rec["cuda_on"] == "rtpose_model"            # model = model.cuda()   (:27)
    monkeypatch.chdir(ROOT)
    glob = _import_as_recorded(rec)
    new_state_dict = {k[6:]: v for k, v in ckpt["state_dict"].items()}
    assert list(new_state_dict) == list(he_sd)
    model = glob["get_model"](trunk="vgg19")                               # (:20-25)
    model.load_state_dict(new_state_dict)
    model = model.eval().float()
    assert type(model).__name__ == rec["cuda_on"]
    assert torch.equal(model.state_dict()["model6_2.12.bias"], he_sd["model6_2.12.bias"])
    inspect.signature(glob["run_eval"]).bind(image_dir="a", anno_file="b", vis_dir="c", model=model, preprocess="vgg")
    assert "OpenPose_Model" in glob and "use_vgg" in glob


@pytest.mark.gpu
def test_demo_with_the_reference_command_line(built, he_sd):
    """`python demo/picture_demo.py` from the repo root, no flags: reads ./experiments/vgg19_368x368_sgd.yaml,
    pose_model.pth and ./readme/ski.jpg, writes result.png - the reference demo's contract (:30-65)."""
    weight, result = os.path.join(ROOT, "pose_model.pth"), os.path.join(ROOT, "result.png")
    torch.save(he_sd, weight)
    try:
        if os.path.exists(result):
            os.remove(result)
        r = subprocess.run([sys.executable, os.path.join("demo", "picture_demo.py")], cwd=ROOT, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True, timeout=600)
        print(r.stdout[-2000:])
        assert r.returncode == 0 and os.path.exists(result)
        assert abs(float(r.stdout.split()[0]) - 368.0 / 674.0) < 1e-12        # print(im_scale)
        assert "humans; maps (46, 49, 19) (46, 49, 38)" in r.stdout           # 674x712 -> 368x389 -> padded 368x392
    finally:
        for f in (weight, result):
            if os.path.exists(f):
                os.remove(f)
