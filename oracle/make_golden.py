"""Generate tests/golden/*.npz by running the UNMODIFIED reference  --  TEST INFRASTRUCTURE ONLY.

Run in the build container only (it needs /root/reference, which does not exist on the
GPU box):

    python oracle/make_golden.py

It imports the reference's own modules (models/editline2_model.py -> EditLine2Model with
netM = MDGenerator, netG = DeepFillC2Generator), loads the seeded synthetic checkpoints of
``sketchedit_b200.synth`` through the reference's strict ``load_state_dict`` and calls the
reference forward ``model(data, mode='inference')`` (reference models/editline2_model.py:107-133)
plus forward hooks on a few inner modules. Nothing from the reference is copied into the
repo: only the numeric inputs/outputs are stored, in the format of ``oracle/golden.py``.
"""
import argparse
import os
import sys
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("SKETCHEDIT_REFERENCE", "/root/reference")


def build_reference_model(flags):
    sys.path.insert(0, REF)
    # the repo's own `models` package mirrors the reference's names: make sure the
    # reference's wins inside this process
    for m in [k for k in sys.modules if k == "models" or k.startswith("models.") or k == "util"
              or k.startswith("util.")]:
        del sys.modules[m]
    from models.editline2_model import EditLine2Model  # noqa: the reference's
    assert os.path.realpath(sys.modules["models"].__file__).startswith(os.path.realpath(REF))
    opt = Namespace(gpu_ids=[], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier",
                    init_variance=0.02, continue_train=False,
                    use_cam=flags.get("use_cam", True), pool_type=flags.get("pool_type", "max"),
                    no_mask_cc=flags.get("no_mask_cc", False),
                    no_mask_coarse=flags.get("no_mask_coarse", False),
                    joint_train_inp=flags.get("joint_train_inp", True))
    model = EditLine2Model(opt)
    model.eval()
    return model


def load_pair(name, release="face_release"):
    from PIL import Image
    img = Image.open(os.path.join(REF, "datasets", release, "images", name)).convert("RGB")
    edge = Image.open(os.path.join(REF, "datasets", release, "edges", name)).convert("L").resize(img.size)
    return np.asarray(img, dtype=np.uint8), np.asarray(edge, dtype=np.uint8)


def u8_case(img_u8, edge_u8, keep=()):
    """reference data/testimage_dataset.py:89-103 preprocessing of a (RGB uint8, L uint8) pair."""
    image = torch.from_numpy(img_u8).permute(2, 0, 1).float().div(255).sub(0.5).div(0.5)[None]
    sketch = (torch.from_numpy(edge_u8).float().div(255) > 0).float()[None, None]
    return dict(inputs=(image, sketch), flags={}, u8=(img_u8, edge_u8), keep=keep)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    ap.add_argument("--only", default=None, help="comma-separated case names (default: all)")
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    from oracle import golden
    from sketchedit_b200 import synth
    torch.set_num_threads(8)
    WM, WG = synth.synth_state_dict("M"), synth.synth_state_dict("G")

    cases = {
        "synth_b2_64x64": dict(inputs=synth.synth_inputs(2, 64, 64, seed=0), flags={}),
        "synth_b1_96x64": dict(inputs=synth.synth_inputs(1, 96, 64, seed=5), flags={}),
        "synth_b1_64x64_avg_nocam": dict(inputs=synth.synth_inputs(1, 64, 64, seed=2),
                                         flags=dict(pool_type="avg", use_cam=False)),
        "synth_b1_64x64_nomask_flags": dict(inputs=synth.synth_inputs(1, 64, 64, seed=3),
                                            flags=dict(no_mask_cc=True, no_mask_coarse=True,
                                                       joint_train_inp=False)),
    }
    # config 1 of BASELINE.json: a real 256x256 face + sketch from the reference's dataset
    cases["face_602_256x256"] = u8_case(*load_pair("602_images_celeb_00033.png"), keep=("fine", "tap:netM.conv_mask_17"))
    # config 4 of BASELINE.json (Places-size contextual attention): the reference's non-square general-scene input,
    # 408 wide x 512 high -> attention over L = 63 * 50 = 3150 patches. Only the end-to-end tensors are kept (file size).
    cases["places_11_512x408"] = u8_case(*load_pair("11.png", "general_release"))
    if args.only:
        cases = {k: v for k, v in cases.items() if k in args.only.split(",")}

    os.makedirs(args.out, exist_ok=True)
    for name, case in cases.items():
        model = build_reference_model(case["flags"])
        model.netM.load_state_dict(WM)           # strict, reference key names
        model.netG.load_state_dict(WG)
        image, sketch = case["inputs"]
        taps = {}

        def hook(key):
            def f(mod, inp, out):
                taps[key] = (out[0] if isinstance(out, tuple) else out).detach().clone()
            return f
        hs = [model.netM.conv10_atrous.register_forward_hook(hook("netM.conv10_atrous")),
              model.netM.conv_mask_17.register_forward_hook(hook("netM.conv_mask_17")),
              model.netG.conv11.register_forward_hook(hook("netG.conv11")),
              model.netG.pmconv6.register_forward_hook(hook("netG.pmconv6")),
              model.netG.cam_2.register_forward_hook(hook("netG.cam")),
              model.netG.allconv16.register_forward_hook(hook("netG.allconv16"))]
        # capture netG's two stage outputs
        stages = {}
        hs.append(model.netG.register_forward_hook(
            lambda m, i, o: stages.update(coarse=o[0].detach().clone(), fine=o[1].detach().clone())))
        data = {"image": image.clone(), "gt": image.clone(), "mask": sketch.clone(),
                "edgegt": sketch.clone()}       # CPU branch needs gt/edgegt supplied (editline2_model.py:225-242)
        with torch.no_grad():
            composed, mask = model(data, mode="inference")
        for h in hs:
            h.remove()
        out = dict(composed=composed.numpy(), mask=mask.numpy(),
                   coarse=stages["coarse"].numpy(), fine=stages["fine"].numpy())
        for k, v in taps.items():
            out["tap:" + k] = v.numpy()
        if "u8" in case:
            inputs = dict(image_u8=case["u8"][0], sketch_u8=case["u8"][1])
            # the real-image cases: only end-to-end tensors (+ what the case asks for)
            out = {k: v for k, v in out.items() if k in ("composed", "mask") + tuple(case["keep"])}
        else:
            inputs = dict(image=image.numpy(), sketch=sketch.numpy())
        path = os.path.join(args.out, name + ".npz")
        golden.save(path, inputs, out, case["flags"])
        print("wrote %s  (%.1f KB)  mask-on %.3f" % (path, os.path.getsize(path) / 1024,
                                                      float((mask > 0.5).float().mean())))


if __name__ == "__main__":
    main()
