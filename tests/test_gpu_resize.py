"""se_resize_u8 on the device against Pillow, byte for byte, and DemoProcessor(resize="device") against the host-resize flow."""
import threading

import numpy as np
import pytest
import torch
from PIL import Image

from sketchedit_b200.engine import resize_u8
from tests.test_resize import SWEEP, sample

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", ["RGB", "L", "mask"])
def test_resize_equals_pillow(kind):
    for i, (src, dst) in enumerate(SWEEP):
        a = sample(kind, *src, seed=100 + i)
        got = resize_u8([torch.from_numpy(a).cuda()], [dst[::-1]])[0].cpu().numpy()
        want = np.array(Image.fromarray(a).resize(dst))
        assert got.shape == want.shape and np.array_equal(got, want), (src, dst)


@pytest.mark.parametrize("channels", [1, 3])
def test_ragged_batch_equals_per_image_calls(channels):
    """One packed batch of every sweep case (gaps between the images, outputs written out of order) == one call per image."""
    kind = "RGB" if channels == 3 else "L"
    imgs = [sample(kind, *src, seed=200 + i) for i, (src, _) in enumerate(SWEEP)]
    src_hw = [a.shape[:2] for a in imgs]
    dst_hw = [dst[::-1] for _, dst in SWEEP]
    src_off = np.concatenate([[0], np.cumsum([a.nbytes + 13 for a in imgs])])
    packed = np.zeros(src_off[-1], np.uint8)
    for a, o in zip(imgs, src_off):
        packed[o:o + a.nbytes] = a.reshape(-1)
    n_out = [h * w * channels for h, w in dst_hw]
    out_off = np.concatenate([[0], np.cumsum(n_out[::-1])])[:-1][::-1]       # last image first
    out = torch.zeros(sum(n_out), dtype=torch.uint8, device="cuda")
    resize_u8(torch.from_numpy(packed).cuda(), dst_hw, src_hw=src_hw, channels=channels, src_offsets=src_off[:-1], out=out,
              out_offsets=out_off)
    out = out.cpu().numpy()
    for a, (h, w), o, n in zip(imgs, dst_hw, out_off, n_out):
        single = resize_u8([torch.from_numpy(a).cuda()], [(h, w)])[0].cpu().numpy()
        assert np.array_equal(out[o:o + n], single.reshape(-1)), (a.shape, (h, w))


def test_reverse_channels():
    for i, (src, dst) in enumerate(SWEEP):
        a = torch.from_numpy(sample("RGB", *src, seed=300 + i)).cuda()
        plain = resize_u8([a], [dst[::-1]])[0]
        rev = resize_u8([a], [dst[::-1]], reverse_channels=True)[0]
        assert torch.equal(rev, plain.flip(-1)), (src, dst)


def test_rejects_out_of_bounds_images():
    from sketchedit_b200._lib import SketchEditB200Error
    buf = torch.zeros(100, dtype=torch.uint8, device="cuda")
    with pytest.raises(SketchEditB200Error, match="outside src"):
        resize_u8(buf, [(4, 4)], src_hw=[(10, 10)], channels=3)
    with pytest.raises(SketchEditB200Error, match="positive"):
        resize_u8(buf, [(0, 4)], src_hw=[(5, 5)], channels=1)


@pytest.mark.parametrize("prec", ["bf16", "fp32_direct"])
def test_device_resize_matches_host_resize(prec):
    """Eight threads, raw sizes that share two floored keys, one mask with a size of its own: resize='device' returns exactly the
    bytes of resize='host'. Every image's forward is bit-identical to its batch-1 run, so batch composition cannot matter."""
    from sketchedit_b200.serving import DemoProcessor
    from tests.test_gpu_configs import _model
    model = _model(prec)
    sizes = [(100, 75), (103, 79), (96, 72), (90, 64), (95, 70), (100, 75), (93, 66), (103, 79)]
    cases = []
    for i, (w, h) in enumerate(sizes):
        m = np.zeros((h, w), np.uint8)
        m[10 + i:40, 20:22 + 3 * i] = 255
        mask = Image.fromarray(m)
        if i == 3:
            mask = mask.resize((w + 9, h - 5))
        cases.append((Image.fromarray(sample("RGB", w, h, seed=400 + i)), mask))
    results = {}
    for mode in ("host", "device"):
        proc = DemoProcessor(model, max_batch=8, max_wait_ms=100.0, resize=mode)
        calls = []
        if mode == "device":     # record the source sizes of every resize call
            proc.engine.resize_u8 = lambda *a, **k: calls.append(k["src_hw"]) or resize_u8(*a, **k)
        got = [None] * len(cases)

        def worker(i):
            got[i] = np.array(proc.process_image(*cases[i]))

        ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(cases))]
        [t.start() for t in ts]
        [t.join() for t in ts]
        proc.close()
        assert {k for k, _ in proc.batcher.batches} == {(72, 96), (64, 88)}
        results[mode] = got
        if mode == "device":
            assert any(len({tuple(hw) for hw in c}) > 1 for c in calls[0::3]), calls       # batches mixed raw sizes
    for (img, _), h, d in zip(cases, results["host"], results["device"]):
        assert h.shape == d.shape == (img.size[1], img.size[0], 3) and np.array_equal(h, d)
