"""CPU oracle and golden vectors of the region inpaint  --  TEST INFRASTRUCTURE ONLY.

``inpaint`` restates, with ``sketchedit_oracle.netG_forward``, the external-mask branch of the reference's generate_fake
(models/editline2_model.py:340-352, 362-368: mask_inpaint = R, line_inpaint = sketch * R, rm2 = R outside training) composed
like :114. netM does not run.

Run as a script in the build container (it needs the reference, like ``oracle/make_golden.py``, whose helpers it uses) to write
``tests/golden/region/*.npz``:

    python oracle/region_oracle.py [--only synth_b2_64x64_region,face_602_256x256_region]

The reference reaches that branch only through ``random.randint`` in training, so the generator calls its ``model.netG(x, x, R, R,
s*R)`` directly and composes like :114. Each file's "mask" output is the region R: the mask netG inpaints and composes with, and
the second output of ``mode='inpaint'``. The files live in a subdirectory because every top-level golden is an input of the netM
path's tests.
"""
import argparse
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.sketchedit_oracle import netG_forward  # noqa: E402


def inpaint(WG, image, sketch, region, **flags):
    """image [B,3,H,W] in [-1,1], sketch and region [B,1,H,W] (region 1 = edit here). Returns dict(composed, coarse, fine)."""
    with torch.no_grad():
        coarse, fine = netG_forward(WG, image, image, region, region, sketch * region, **flags)
        composed = fine * region + image * (1 - region)
    return dict(composed=composed, coarse=coarse, fine=fine)


def synth_regions(B, H, W, seed):
    """[B,1,H,W] 0/1: a seeded rectangle and ellipse per image; the last image's region is empty."""
    rs = np.random.RandomState(seed)
    R = np.zeros((B, 1, H, W), np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    for b in range(B - 1):
        y0, x0 = rs.randint(0, H // 2), rs.randint(0, W // 2)
        R[b, 0, y0:y0 + rs.randint(H // 4, H // 2), x0:x0 + rs.randint(W // 4, W // 2)] = 1
        cy, cx, ry, rx = rs.randint(H // 4, 3 * H // 4), rs.randint(W // 4, 3 * W // 4), rs.randint(4, H // 4), rs.randint(4, W // 4)
        R[b, 0][((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1] = 1
    return torch.from_numpy(R)


def main():
    from oracle import golden
    from oracle import make_golden as G
    from sketchedit_b200 import synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "region"))
    ap.add_argument("--only", default=None, help="comma-separated case names (default: all)")
    args = ap.parse_args()
    torch.set_num_threads(8)
    WG = synth.synth_state_dict("G")
    # seeded shapes on synthetic inputs (one image with an empty region); the 602 face with a user circling its strokes, i.e. the
    # sketch dilated by a 31x31 box
    image, sketch = synth.synth_inputs(2, 64, 64, seed=7)
    R = synth_regions(2, 64, 64, seed=7)
    cases = {"synth_b2_64x64_region": dict(image=image, sketch=sketch, region=R,
                                           inputs=dict(image=image.numpy(), sketch=sketch.numpy(), region=R.numpy()))}
    face = G.u8_case(*G.load_pair("602_images_celeb_00033.png"))
    dil = torch.nn.functional.max_pool2d(torch.from_numpy(face["u8"][1] > 0).float()[None, None], 31, stride=1, padding=15)
    region_u8 = (dil[0, 0].numpy() > 0).astype(np.uint8) * 255
    cases["face_602_256x256_region"] = dict(image=face["inputs"][0], sketch=face["inputs"][1],
                                            region=torch.from_numpy(region_u8 > 0).float()[None, None],
                                            inputs=dict(image_u8=face["u8"][0], sketch_u8=face["u8"][1], region_u8=region_u8))
    if args.only:
        cases = {k: v for k, v in cases.items() if k in args.only.split(",")}
    os.makedirs(args.out, exist_ok=True)
    for name, case in cases.items():
        model = G.build_reference_model({})
        model.netG.load_state_dict(WG)           # strict, reference key names
        x, s, R = case["image"], case["sketch"], case["region"]
        with torch.no_grad():
            coarse, fine = model.netG(x, x, R, R, s * R)
            composed = fine * R + x * (1 - R)
        out = dict(composed=composed.numpy(), mask=R.numpy(), coarse=coarse.numpy(), fine=fine.numpy())
        path = os.path.join(args.out, name + ".npz")
        golden.save(path, case["inputs"], out, {})
        print("wrote %s  (%.1f KB)  region %.3f" % (os.path.relpath(path, ROOT), os.path.getsize(path) / 1024, float(R.mean())))


if __name__ == "__main__":
    main()
