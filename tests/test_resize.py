"""Pillow-exact resize of the serving path, host side (no GPU): the numpy restatement against the installed Pillow, the library's
coefficient tables against the restatement, and DemoProcessor's ragged packing with a fake engine."""
import threading

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import pil_resample as R
from sketchedit_b200 import _lib, build
from sketchedit_b200.serving import DemoProcessor

# (width, height) in -> out, as PIL takes them: the demo's 637x477 request, both directions of a small pair, one axis only,
# halving with an odd source, growing by non-integer factors, tiny sizes, a 1-pixel-wide source, the same size
SWEEP = [((637, 477), (632, 472)), ((632, 472), (637, 477)), ((100, 75), (96, 72)), ((96, 72), (100, 75)), ((90, 64), (88, 64)),
         ((64, 90), (64, 88)), ((513, 300), (256, 150)), ((40, 30), (123, 97)), ((17, 9), (16, 8)), ((1, 5), (8, 8)), ((50, 40), (50, 40))]


def sample(kind, w, h, seed):
    rs = np.random.RandomState(seed)
    if kind == "RGB":
        return rs.randint(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "L":
        return rs.randint(0, 256, (h, w), dtype=np.uint8)
    return (rs.rand(h, w) > 0.8).astype(np.uint8) * 255          # binary sketch mask


@pytest.mark.parametrize("kind", ["RGB", "L", "mask"])
@pytest.mark.parametrize("src,dst", SWEEP)
def test_restatement_equals_pillow(src, dst, kind):
    a = sample(kind, *src, seed=src[0] * 7 + dst[1])
    want = np.array(Image.fromarray(a).resize(dst))
    got = R.resize(a, dst)
    assert got.shape == want.shape and np.array_equal(got, want)


@pytest.fixture(scope="module")
def lib():
    build.build(verbose=False)
    return _lib.load()


def test_library_coefficient_tables_equal_the_restatement(lib):
    pairs = {(s[i], d[i]) for s, d in SWEEP for i in (0, 1) if s[i] != d[i]} | {(1000, 13), (3, 1)}
    for n_in, n_out in sorted(pairs):
        ksize = lib.se_resize_coeffs(n_in, n_out, None, None, 0)
        bounds, weights = np.zeros((n_out, 2), np.int32), np.zeros((n_out, ksize), np.int32)
        assert lib.se_resize_coeffs(n_in, n_out, bounds.ctypes.data, weights.ctypes.data, weights.size) == ksize
        want_b, want_w = R.coeffs(n_in, n_out)
        assert np.array_equal(bounds, want_b) and np.array_equal(weights, want_w), (n_in, n_out)
    assert lib.se_resize_coeffs(0, 8, None, None, 0) == -1 and b"positive" in lib.se_last_error()


class FakeEngine:
    """Stands in for Engine on the CPU: resize_u8 (packed form) through the numpy restatement, and a forward that is a fixed
    per-image function of its uint8 inputs, so a request's result does not depend on its batch (as the real one's does not)."""
    device = torch.device("cpu")

    def __init__(self):
        self.resize_calls = []

    def resize_u8(self, src, dst_hw, src_hw=None, channels=None, src_offsets=None, reverse_channels=False):
        self.resize_calls.append([tuple(int(v) for v in hw) for hw in src_hw])
        flat, outs = src.reshape(-1).numpy(), []
        if src_offsets is None:
            src_offsets = np.concatenate([[0], np.cumsum([h * w * channels for h, w in src_hw])])[:-1]
        for (h, w), o, (ho, wo) in zip(src_hw, src_offsets, dst_hw):
            a = flat[o:o + h * w * channels].reshape((h, w, channels) if channels > 1 else (h, w))
            r = R.resize(a, (wo, ho))
            outs.append((r[..., ::-1] if reverse_channels else r).reshape(-1))
        return torch.from_numpy(np.concatenate(outs))

    @staticmethod
    def forward(img, mask):
        """[H,W,3] RGB, [H,W] (> 0 = sketch) -> [H,W,3] BGR"""
        out = img.astype(np.int32) * 3 + (mask > 0)[..., None] * 101 + np.arange(3) * 17
        return (out % 256).astype(np.uint8)[..., ::-1]

    def inference_u8(self, img, mask, precision):
        bgr = np.stack([self.forward(i, m) for i, m in zip(img.numpy(), mask.numpy())])
        return torch.from_numpy(np.ascontiguousarray(bgr)), None


class FakeModel:
    precision = "bf16"

    def __init__(self):
        self.eng = FakeEngine()

    def engine(self):
        return self.eng


def test_device_mode_packs_ragged_batches_and_splits_results():
    """Raw sizes that floor to one size share a batch; each request gets Pillow-resize-back(forward(Pillow-resize-in(image),
    Pillow-resize-in(mask) > 0)) at its own size, whichever batch it rode in. One mask has a size of its own."""
    sizes = [(100, 75), (103, 79), (96, 72), (90, 64), (95, 70), (100, 75), (93, 66), (103, 79)]
    cases = []
    for i, (w, h) in enumerate(sizes):
        mw, mh = (w + 9, h - 5) if i == 3 else (w, h)
        cases.append((Image.fromarray(sample("RGB", w, h, seed=i)), Image.fromarray(sample("mask", mw, mh, seed=50 + i))))
    model = FakeModel()
    proc = DemoProcessor(model, max_batch=8, max_wait_ms=200.0, resize="device")
    got = [None] * len(cases)

    def worker(i):
        got[i] = proc.process_image(*cases[i])

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(len(cases))]
    [t.start() for t in ts]
    [t.join() for t in ts]
    proc.close()
    assert {k for k, _ in proc.batcher.batches} == {(72, 96), (64, 88)} and len(proc.batcher.batches) < len(cases)
    image_calls = model.eng.resize_calls[0::3]                  # per batch: images in, masks in, results out
    assert any(len(set(c)) > 1 for c in image_calls)             # a batch really held several raw sizes
    for (img, mask), res in zip(cases, got):
        w, h = img.size
        key = (w // 8 * 8, h // 8 * 8)
        bgr = FakeEngine.forward(np.array(img.resize(key)), np.array(mask.resize(key)))
        want = np.array(Image.fromarray(np.ascontiguousarray(bgr[..., ::-1])).resize((w, h)))
        assert res.size == (w, h) and np.array_equal(np.array(res), want)


def test_device_mode_rejects_a_mask_that_is_not_L():
    proc = DemoProcessor(FakeModel(), resize="device")
    with pytest.raises(ValueError, match="'L'"):
        proc.process_image(Image.new("RGB", (64, 64)), Image.new("1", (64, 64)))
    proc.close()
    with pytest.raises(ValueError):
        DemoProcessor(FakeModel(), resize="gpu")
