"""GPU parity of netM / netG / the whole inference path against the CPU oracle and the committed
reference-generated golden vectors.

Tolerances are BASELINE.json's: 1e-3 max-abs (fp32 path), 1e-2 (bf16 tensor-core path), both against
the fp32 oracle. The mask threshold (reference editline2_model.py:347) is discontinuous, so netG and the
end-to-end output are compared with the oracle evaluated on OUR binarised mask; the number of
threshold flips against the oracle's own mask is bounded separately (SURVEY.md section 7.3-2).
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import sketchedit_oracle as O
from oracle.golden import Golden
from sketchedit_b200 import synth
from tests.util_parity import engine, maxdiff, weights

pytestmark = pytest.mark.gpu
TOL = {"fp32": 1e-3, "fp32_direct": 1e-3, "bf16": 1e-2}   # "fp32": split-half tensor-core arithmetic, "fp32_direct": CUDA cores


@pytest.mark.parametrize("prec", ["fp32", "fp32_direct", "bf16"])
def test_netM(prec):
    WM, _ = weights()
    img, sk = synth.synth_inputs(2, 64, 96, seed=11)
    mask, st1 = engine().netM(img.cuda(), sk.cuda(), precision=prec)
    rm, rs = O.netM_forward(WM, img, sk)
    assert maxdiff(mask.cpu(), rm) <= TOL[prec]
    assert maxdiff(st1.cpu(), rs) <= TOL[prec]


@pytest.mark.parametrize("prec", ["fp32", "fp32_direct", "bf16"])
def test_netG(prec):
    _, WG = weights()
    img, sk = synth.synth_inputs(2, 64, 64, seed=12)
    mask = torch.zeros(2, 1, 64, 64)
    mask[0, :, 16:40, 8:50] = 1
    mask[1, :, 30:60, 20:44] = 1
    s1, s2 = engine().netG(img.cuda(), img.cuda(), mask.cuda(), mask.cuda(), sk.cuda(), precision=prec)
    r1, r2 = O.netG_forward(WG, img, img, mask, mask, sk)
    assert maxdiff(s1.cpu(), r1) <= TOL[prec], maxdiff(s1.cpu(), r1)
    assert maxdiff(s2.cpu(), r2) <= TOL[prec], maxdiff(s2.cpu(), r2)


@pytest.mark.parametrize("prec", ["fp32", "fp32_direct", "bf16"])
@pytest.mark.parametrize("shape", [(2, 64, 64), (1, 96, 64), (1, 128, 104)])
def test_inference_vs_oracle(prec, shape):
    WM, WG = weights()
    B, H, W = shape
    img, sk = synth.synth_inputs(B, H, W, seed=H + W)
    composed, mask, ex = engine().inference(img.cuda(), sk.cuda(), precision=prec, want=("coarse", "fine", "mask_bin"))
    ours_bin = ex["mask_bin"].cpu()
    ref_free = O.inference(WM, WG, img, sk)
    flips = int((ours_bin != ref_free["mask_bin"]).sum())
    assert flips <= (0 if prec.startswith("fp32") else 0.02 * ours_bin.numel()), flips
    ref = O.inference(WM, WG, img, sk, mask_bin_override=ours_bin)
    assert maxdiff(mask.cpu(), ref["mask"]) <= TOL[prec]
    for k, t in (("coarse", ex["coarse"]), ("fine", ex["fine"]), ("composed", composed)):
        assert maxdiff(t.cpu(), ref[k]) <= TOL[prec], (k, maxdiff(t.cpu(), ref[k]))


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in
                                        glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))))
@pytest.mark.parametrize("prec", ["fp32", "fp32_direct"])
def test_fp32_path_matches_reference_golden(name, golden_dir, prec):
    """fp32 paths (tensor-core split-half arithmetic and the CUDA-core cross-check) vs outputs of the unmodified reference
    (tests/golden, oracle/make_golden.py)."""
    g = Golden(os.path.join(golden_dir, name + ".npz"))
    image, sketch = g.inputs()
    eng = engine(**g.flags)
    composed, mask, ex = eng.inference(image.cuda(), sketch.cuda(), precision=prec, want=("fine", "mask_bin"))
    assert int((ex["mask_bin"].cpu() != g.mask_bin()).sum()) == 0
    assert g.maxdiff("mask", mask) <= 1e-3
    if "fine" in g:
        assert g.maxdiff("fine", ex["fine"]) <= 1e-3
    assert g.maxdiff("composed", composed) <= 1e-3


def test_bf16_face_config(golden_dir):
    """BASELINE.json config: 256x256 face + sketch, bf16 tensor-core path, 1e-2 vs the fp32 reference."""
    WM, WG = weights()
    g = Golden(os.path.join(golden_dir, "face_602_256x256.npz"))
    image, sketch = g.inputs()
    composed, mask, ex = engine().inference(image.cuda(), sketch.cuda(), precision="bf16", want=("mask_bin",))
    assert g.maxdiff("mask", mask) <= 1e-2
    ours_bin = ex["mask_bin"].cpu()
    ref = O.inference(WM, WG, image, sketch, mask_bin_override=ours_bin)
    assert maxdiff(composed.cpu(), ref["composed"]) <= 1e-2


def test_batch_sharding_is_exact():
    """Per-sample independence (SURVEY.md section 8e): forward(batch)[i] == forward(batch[i:i+1]) bit for bit."""
    img, sk = synth.synth_inputs(3, 64, 64, seed=5)
    eng = engine()
    full, fm, _ = eng.inference(img.cuda(), sk.cuda(), precision="bf16")
    for i in range(3):
        one, om, _ = eng.inference(img[i:i + 1].cuda(), sk[i:i + 1].cuda(), precision="bf16")
        assert torch.equal(one[0], full[i]) and torch.equal(om[0], fm[i])


def test_uint8_outputs():
    from sketchedit_b200.engine import outputs_to_uint8
    img, sk = synth.synth_inputs(1, 64, 64, seed=9)
    composed, mask, _ = engine().inference(img.cuda(), sk.cuda(), precision="bf16")
    bgr, mk = outputs_to_uint8(composed, mask)
    g, m = O.to_uint8_outputs(composed.cpu(), mask.cpu())
    assert np.array_equal(bgr.cpu().numpy(), g.transpose(0, 2, 3, 1)[..., ::-1])
    assert np.array_equal(mk.cpu().numpy(), m)


def test_inference_stream_matches_blocking_calls():
    """models.EditLine2Model.inference_stream (copies on side streams, double-buffered) returns, in order and bit for
    bit, what one blocking model(data, mode='inference') call per batch returns - including a ragged last batch."""
    from argparse import Namespace

    import models
    opt = Namespace(gpu_ids=[0], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02,
                    use_cam=True, pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True,
                    model="editline2", precision="bf16")
    model = models.create_model(opt)
    model.netM.load_state_dict(synth.synth_state_dict("M"))
    model.netG.load_state_dict(synth.synth_state_dict("G"))
    model.eval()
    batches = []
    for i, b in enumerate((2, 2, 2, 2, 1)):
        img, sk = synth.synth_inputs(b, 64, 64, seed=20 + i)
        batches.append({"image": img.pin_memory(), "mask": sk.pin_memory()})
    with torch.no_grad():
        want = [tuple(t.cpu() for t in model(d, mode="inference")) for d in batches]
        got = [(c.clone(), m.clone()) for c, m in model.inference_stream(iter(batches))]   # results are ring views
        fresh = list(model.inference_stream(iter(batches), pinned_ring=False))
    assert len(got) == len(want)
    for (gc, gm), (fc, fm), (wc, wm) in zip(got, fresh, want):
        assert torch.equal(gc, wc) and torch.equal(gm, wm)
        assert fc.is_pinned() and torch.equal(fc, wc) and torch.equal(fm, wm)
