"""Region inpaint, host side (no GPU): the CPU oracle against the unmodified reference's netG on user regions
(tests/golden/region/*.npz, oracle/region_oracle.py), and DemoProcessor's region requests with a fake engine."""
import glob
import os
import threading
from argparse import Namespace

import numpy as np
import pytest
import torch
from PIL import Image

from oracle.region_oracle import inpaint
from oracle.golden import Golden
from sketchedit_b200 import synth
from sketchedit_b200.serving import DemoProcessor
from tests.test_resize import FakeEngine, sample

TOL = 2e-5   # fp32 vs fp32, as tests/test_oracle_golden.py
REGION_GOLDEN = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "region", "*.npz")))


def region_inputs(g):
    """(image, sketch, region) of a region golden; uint8 files decode the region like the sketch (> 0)."""
    image, sketch = g.inputs()
    if "region" in g.z:
        return image, sketch, torch.from_numpy(g.z["region"])
    return image, sketch, (torch.from_numpy(g.z["region_u8"]) > 0).float()[None, None]


def test_region_goldens_exist():
    assert REGION_GOLDEN == ["face_602_256x256_region", "synth_b2_64x64_region"]


@pytest.mark.parametrize("name", REGION_GOLDEN)
def test_oracle_inpaint_matches_reference(name, golden_dir):
    WG = synth.synth_state_dict("G")
    g = Golden(os.path.join(golden_dir, "region", name + ".npz"))
    image, sketch, region = region_inputs(g)
    assert torch.equal(g.mask_bin(), region)         # the stored "mask" is the region netG inpainted and composed with
    r = inpaint(WG, image, sketch, region, **g.flags)
    for key in ("composed", "coarse", "fine"):
        d = g.maxdiff(key, r[key])
        assert d <= TOL, (name, key, d)
    assert torch.equal(r["composed"] * (1 - region), image * (1 - region))


def test_model_inpaint_needs_a_region():
    import models
    opt = Namespace(gpu_ids=[], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02, use_cam=True,
                    pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True, model="editline2", precision="bf16")
    model = models.create_model(opt)
    with pytest.raises(KeyError, match="region"):
        model({"image": torch.zeros(1, 3, 64, 64), "mask": torch.zeros(1, 1, 64, 64)}, mode="inpaint")


# ------------------------------------------------------------------------------------------------ serving
class RegionFakeEngine(FakeEngine):
    """FakeEngine plus a region forward that is a fixed per-image function of (image, sketch > 0, region > 0), distinct from the
    plain forward, so a result shows which forward and which planes produced it."""

    def __init__(self):
        super().__init__()
        self.forwards = []

    @staticmethod
    def forward_region(img, mask, region):
        r = (region > 0)[..., None]
        return np.where(r, FakeEngine.forward(img, mask)[..., ::-1] ^ 0x5A, img).astype(np.uint8)[..., ::-1]

    def inference_u8(self, img, mask, precision):
        self.forwards.append(("plain", tuple(img.shape)))
        return super().inference_u8(img, mask, precision)

    def inpaint_u8(self, img, mask, region, precision):
        self.forwards.append(("region", tuple(img.shape)))
        bgr = np.stack([self.forward_region(i, m, r) for i, m, r in zip(img.numpy(), mask.numpy(), region.numpy())])
        return torch.from_numpy(np.ascontiguousarray(bgr))


class FakeModel:
    precision = "bf16"

    def __init__(self):
        self.eng = RegionFakeEngine()

    def engine(self):
        return self.eng


@pytest.mark.parametrize("resize", ["host", "device"])
def test_region_requests_batch_apart_and_route_back(resize):
    """Plain and region requests of the same sizes from many threads: a batch never mixes them, region batches carry the key
    (h, w, "region"), plain ones keep (h, w), the region is resized and binarised exactly like the sketch, and every caller gets
    the result of its own request. One region (device mode: also one sketch) has a size of its own."""
    sizes = [(100, 75), (103, 79), (96, 72), (90, 64), (95, 70), (100, 75), (93, 66), (103, 79)]
    cases = []
    for i, (w, h) in enumerate(sizes * 2):
        img = Image.fromarray(sample("RGB", w, h, seed=i))
        mask = Image.fromarray(sample("mask", w, h, seed=50 + i))
        region = None
        if i % 2:
            rw, rh = (w - 7, h + 4) if i == 5 else (w, h)
            region = Image.fromarray(sample("L", rw, rh, seed=90 + i) // 2)       # values 0..127: binarised as > 0, not > 127
        cases.append((img, mask, region))
    model = FakeModel()
    proc = DemoProcessor(model, max_batch=8, max_wait_ms=200.0, resize=resize)
    got = [None] * len(cases)

    def worker(i):
        got[i] = proc.process_image(*cases[i])

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(cases))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    proc.close()
    keys = {k for k, _ in proc.batcher.batches}
    assert keys == {(72, 96), (64, 88), (72, 96, "region"), (64, 88, "region")}
    assert sum(n for _, n in proc.batcher.batches) == len(cases) and len(proc.batcher.batches) < len(cases)
    kinds = [k for k, _ in model.eng.forwards]
    assert kinds == ["region" if len(k) == 3 else "plain" for k, _ in proc.batcher.batches]
    for (img, mask, region), res in zip(cases, got):
        w, h = img.size
        size = (w // 8 * 8, h // 8 * 8)
        im, sk = np.array(img.resize(size)), np.array(mask.resize(size)) > 0
        if region is None:
            bgr = FakeEngine.forward(im, sk)
        else:
            bgr = RegionFakeEngine.forward_region(im, sk, np.array(region.resize(size)) > 0)
        want = np.array(Image.fromarray(np.ascontiguousarray(bgr[..., ::-1])).resize((w, h)))
        assert res.size == (w, h) and np.array_equal(np.array(res), want)


def test_device_mode_rejects_a_region_that_is_not_L():
    proc = DemoProcessor(FakeModel(), resize="device")
    with pytest.raises(ValueError, match="'L'"):
        proc.process_image(Image.new("RGB", (64, 64)), Image.new("L", (64, 64)), Image.new("1", (64, 64)))
    proc.close()
