"""Region inpaint on the GPU (se_forward_inpaint / se_forward_inpaint_u8): parity with the CPU oracle and with the unmodified
reference's netG on user regions (tests/golden/region), the image kept exactly outside the region, the uint8 codecs, batch and
CUDA-graph invariance, netM skipped, the module surface and the demo flow.

Tolerances are BASELINE's: 1e-3 max-abs for the fp32 modes, 1e-2 for bf16. netG sees the caller's region, so there is no threshold
and no flip allowance."""
import ctypes
import json
import os
import threading

import numpy as np
import pytest
import torch
from PIL import Image

from oracle.region_oracle import inpaint
from oracle.golden import Golden
from sketchedit_b200 import _lib, synth
from tests.test_inpaint import REGION_GOLDEN, region_inputs
from tests.util_parity import engine, maxdiff, weights

pytestmark = pytest.mark.gpu
TOL = {"fp32": 1e-3, "fp32_direct": 1e-3, "bf16": 1e-2}
PRECS = ["fp32", "fp32_direct", "bf16"]


def regions(B, H, W, seed, empty_last=False):
    """[B,1,H,W] 0/1: a seeded rectangle and ellipse per image (the last one empty if asked)."""
    rs = np.random.RandomState(seed)
    R = np.zeros((B, 1, H, W), np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    for b in range(B - 1 if empty_last else B):
        y0, x0 = rs.randint(0, H // 2), rs.randint(0, W // 2)
        R[b, 0, y0:y0 + rs.randint(H // 4, H // 2), x0:x0 + rs.randint(W // 4, W // 2)] = 1
        cy, cx, ry, rx = rs.randint(H // 4, 3 * H // 4), rs.randint(W // 4, 3 * W // 4), rs.randint(4, H // 4), rs.randint(4, W // 4)
        R[b, 0][((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1] = 1
    return torch.from_numpy(R)


def u8_inputs(B, H, W, seed):
    rs = np.random.RandomState(seed)
    img = torch.from_numpy(rs.randint(0, 256, (B, H, W, 3), dtype=np.uint8))
    sk = torch.from_numpy((rs.rand(B, H, W) > 0.97).astype(np.uint8) * rs.randint(1, 256, (B, H, W)).astype(np.uint8))
    rg = (regions(B, H, W, seed + 1)[:, 0] * torch.from_numpy(rs.randint(1, 256, (B, H, W)).astype(np.float32))).to(torch.uint8)
    return img, sk, rg


def decode(img_u8, sk_u8, rg_u8):
    """the reference's dataset codec (data/testimage_dataset.py:89-103) on the host; the region decodes like the sketch"""
    image = img_u8.permute(0, 3, 1, 2).float().div(255).sub(0.5).div(0.5)
    return image, (sk_u8.float().div(255)[:, None] > 0).float(), (rg_u8.float().div(255)[:, None] > 0).float()


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("shape", [(2, 64, 64), (1, 96, 64), (1, 128, 104)])
def test_inpaint_vs_oracle(prec, shape):
    _, WG = weights()
    B, H, W = shape
    img, sk = synth.synth_inputs(B, H, W, seed=H + W + 1)
    R = regions(B, H, W, seed=H * W)
    composed, ex = engine().inpaint(img.cuda(), sk.cuda(), R.cuda(), precision=prec, want=("coarse", "fine"))
    ref = inpaint(WG, img, sk, R)
    for k, t in (("coarse", ex["coarse"]), ("fine", ex["fine"]), ("composed", composed)):
        assert maxdiff(t.cpu(), ref[k]) <= TOL[prec], (k, maxdiff(t.cpu(), ref[k]))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", REGION_GOLDEN)
def test_inpaint_matches_reference_golden(name, prec, golden_dir):
    g = Golden(os.path.join(golden_dir, "region", name + ".npz"))
    image, sketch, region = region_inputs(g)
    composed, ex = engine(**g.flags).inpaint(image.cuda(), sketch.cuda(), region.cuda(), precision=prec, want=("coarse", "fine"))
    for k, t in (("coarse", ex["coarse"]), ("fine", ex["fine"]), ("composed", composed)):
        assert g.maxdiff(k, t) <= TOL[prec], (k, g.maxdiff(k, t))
    out = (region == 0).expand_as(image)
    assert torch.equal(composed.cpu()[out], image[out])


@pytest.mark.parametrize("prec", PRECS)
def test_image_kept_exactly_outside_the_region(prec):
    img, sk = synth.synth_inputs(2, 64, 96, seed=71)
    R = regions(2, 64, 96, seed=72, empty_last=True)
    composed, _ = engine().inpaint(img.cuda(), sk.cuda(), R.cuda(), precision=prec)
    out = (R == 0).expand_as(img)
    assert torch.equal(composed.cpu()[out], img[out])
    assert torch.equal(composed[1].cpu(), img[1])                                     # R == 0 everywhere: the whole image
    zero, _ = engine().inpaint(img.cuda(), sk.cuda(), torch.zeros_like(R).cuda(), precision=prec)
    assert torch.equal(zero.cpu(), img)


@pytest.mark.parametrize("prec", PRECS)
def test_uint8_entry_equals_float_entry(prec):
    """inpaint_u8 (input codec kernel, output codec fused into the last head) == the float entry on host-decoded inputs followed by
    outputs_to_uint8, byte for byte."""
    from sketchedit_b200.engine import outputs_to_uint8
    img_u8, sk_u8, rg_u8 = u8_inputs(2, 64, 96, seed=81)
    eng = engine()
    bgr = eng.inpaint_u8(img_u8.cuda(), sk_u8.cuda(), rg_u8.cuda(), precision=prec)
    image, sketch, region = decode(img_u8, sk_u8, rg_u8)
    composed, _ = eng.inpaint(image.cuda(), sketch.cuda(), region.cuda(), precision=prec)
    want, _ = outputs_to_uint8(composed, region.cuda())
    assert torch.equal(bgr, want)


def test_batch_independence_and_graph_replay():
    """bf16 256x256 batch 32: every image equals its batch-1 run bit for bit; three calls with the same buffers (eager, captured,
    replayed) give the same bytes, in both entries."""
    B, H, W = 32, 256, 256
    img_u8, sk_u8, rg_u8 = (t.cuda() for t in u8_inputs(B, H, W, seed=91))
    image, sketch, region = (t.cuda() for t in decode(img_u8.cpu(), sk_u8.cpu(), rg_u8.cpu()))
    eng = engine()
    full, _ = eng.inpaint(image, sketch, region, precision="bf16")
    for i in range(B):
        one, _ = eng.inpaint(image[i:i + 1], sketch[i:i + 1], region[i:i + 1], precision="bf16")
        assert torch.equal(one[0], full[i]), i
    out = torch.empty(B, H, W, 3, dtype=torch.uint8, device="cuda")
    got = [eng.inpaint_u8(img_u8, sk_u8, rg_u8, precision="bf16", out=out).clone() for _ in range(3)]
    assert torch.equal(got[0], got[1]) and torch.equal(got[1], got[2])
    outf = torch.empty(B, 3, H, W, device="cuda")
    gotf = [eng.inpaint(image, sketch, region, precision="bf16", out=outf)[0].clone() for _ in range(3)]
    assert torch.equal(gotf[0], full) and torch.equal(gotf[1], full) and torch.equal(gotf[2], full)


def _classes(run):
    lib = _lib.load()
    lib.se_timing_enable(1)
    try:
        run()
        torch.cuda.synchronize()
        buf = ctypes.create_string_buffer(1 << 20)
        _lib.check(0 if lib.se_timing_report(buf, len(buf)) >= 0 else 1)
        return [c["name"] for c in json.loads(buf.value.decode())["classes"]]
    finally:
        lib.se_timing_enable(0)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_netM_does_not_run(prec):
    """One instrumented call: no netM layer class. netM alone has a 4-channel 5x5 stem (image + sketch) and a 1-channel head
    (sigmoid + threshold); the inference call shows both, the inpaint call neither, and it launches fewer kernels."""
    img, sk = synth.synth_inputs(2, 64, 64, seed=101)
    R = regions(2, 64, 64, seed=102).cuda()
    eng = engine()
    netM_class = lambda n: " 4->48 k5" in n or "12->1 " in n or "sigmoid" in n
    inf = _classes(lambda: eng.inference(img.cuda(), sk.cuda(), precision=prec))
    n_inf = eng.launches()
    inp = _classes(lambda: eng.inpaint(img.cuda(), sk.cuda(), R, precision=prec))
    n_inp = eng.launches()
    assert sum(map(netM_class, inf)) == 2, inf
    assert not any(map(netM_class, inp)), inp
    assert any(n.startswith("region_inputs_kernel") for n in inp), inp
    assert n_inp < n_inf, (n_inp, n_inf)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_model_inpaint_mode(prec):
    from tests.test_gpu_configs import _model
    img, sk = synth.synth_inputs(2, 64, 96, seed=111)
    R = regions(2, 64, 96, seed=112)
    model = _model(prec)
    with torch.no_grad():
        composed, region = model({"image": img, "mask": sk, "region": R}, mode="inpaint")
    want, _ = model.engine().inpaint(img.cuda(), sk.cuda(), R.cuda(), precision=prec)
    assert torch.equal(composed, want) and torch.equal(region.cpu(), R)


def _demo_cases(n, seed):
    """(image, sketch, region) PIL triples at raw sizes that floor to two network sizes; one region has a size of its own"""
    rs = np.random.RandomState(seed)
    sizes = [(100, 75), (103, 79), (96, 72), (90, 64), (95, 70), (100, 75), (93, 66), (103, 79)]
    cases = []
    for i in range(n):
        w, h = sizes[i % len(sizes)]
        img = Image.fromarray(rs.randint(0, 256, (h, w, 3), dtype=np.uint8))
        m = np.zeros((h, w), np.uint8)
        m[10 + i:40, 20:22 + 3 * i] = 255
        r = np.zeros((h, w), np.uint8)
        r[5 + i:50, 12:30 + 3 * i] = 200
        region = Image.fromarray(r)
        if i == 3:
            region = region.resize((w + 9, h - 5))
        cases.append((img, Image.fromarray(m), region))
    return cases


@pytest.mark.parametrize("prec", ["bf16", "fp32_direct"])
def test_demo_regions_device_resize_matches_host_resize(prec):
    """Eight threads, mixed raw sizes, region and plain requests interleaved: resize='device' returns exactly the bytes of
    resize='host', and region requests batch under (h, w, "region")."""
    from sketchedit_b200.serving import DemoProcessor
    from tests.test_gpu_configs import _model
    model = _model(prec)
    cases = _demo_cases(8, seed=121)
    results = {}
    for mode in ("host", "device"):
        proc = DemoProcessor(model, max_batch=8, max_wait_ms=100.0, resize=mode)
        got = [None] * len(cases)

        def worker(i):
            img, m, r = cases[i]
            got[i] = np.array(proc.process_image(img, m, r if i % 4 else None))

        ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(cases))]
        [t.start() for t in ts]
        [t.join() for t in ts]
        proc.close()
        assert {k for k, _ in proc.batcher.batches} == {(72, 96), (64, 88), (72, 96, "region"), (64, 88, "region")}
        results[mode] = got
    for (img, _, _), h, d in zip(cases, results["host"], results["device"]):
        assert h.shape == d.shape == (img.size[1], img.size[0], 3) and np.array_equal(h, d)


def test_demo_regions_match_the_reference_demo_flow():
    """process_image with a region == the reference demo's steps (demo.py:39-73: floor to a multiple of 8, PIL resize, codec,
    forward, clamp, (g+1)/2*255 truncated, PIL resize back) around the oracle's region inpaint, within the bound of
    test_process_image_matches_the_reference_demo_flow."""
    from sketchedit_b200.serving import DemoProcessor
    from tests.test_gpu_configs import _model
    model = _model("fp32_direct")
    proc = DemoProcessor(model, max_batch=4, max_wait_ms=50.0)
    _, WG = weights()
    cases = _demo_cases(8, seed=131)
    got = [None] * len(cases)

    def worker(i):
        got[i] = proc.process_image(*cases[i])

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(cases))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    proc.close()
    assert {k for k, _ in proc.batcher.batches} == {(72, 96, "region"), (64, 88, "region")}
    for (img, mask, region), res in zip(cases, got):
        w_raw, h_raw = img.size
        h_t, w_t = h_raw // 8 * 8, w_raw // 8 * 8
        it = torch.from_numpy(np.array(img.resize((w_t, h_t))).transpose(2, 0, 1)).float()
        it = ((it / 255 - 0.5) / 0.5)[None]
        mt = (torch.from_numpy(np.array(mask.resize((w_t, h_t)))).float() > 0).float()[None, None]
        rt = (torch.from_numpy(np.array(region.resize((w_t, h_t)))).float() > 0).float()[None, None]
        ref = inpaint(WG, it, mt, rt)["composed"]
        ref = ((torch.clamp(ref, -1, 1) + 1) / 2 * 255).numpy().astype(np.uint8)[0].transpose(1, 2, 0)
        want = np.array(Image.fromarray(ref).resize((w_raw, h_raw)))
        assert res.size == (w_raw, h_raw)
        d = np.abs(np.array(res).astype(int) - want.astype(int))
        assert d.max() <= 2 and (d != 0).mean() <= 5e-3, (d.max(), (d != 0).mean())
