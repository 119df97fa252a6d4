"""Serving side of the reference's second entry point (reference demo.py:39-73, SURVEY.md 8f-3), without the Flask UI.

The reference's demo handles one request per Flask thread (``app.run(threaded=True)``) and every request runs its own
batch-1 forward. Here concurrent requests are BATCHED: ``RequestBatcher`` collects the requests that arrive within a short
window, groups them by input size and runs each group as one forward (``Engine.inference_u8``: the codecs of
demo.py:52-53,64-66 run on the device); ``DemoProcessor.process_image`` is the reference's ``process_image`` around it
(floor the size to a multiple of 8, PIL resize in, forward, PIL resize back). With ``resize="device"`` the three resizes run
on the device too (``engine.resize_u8``, bit for bit Pillow's), so one batch holds every raw size that floors to its key.

    proc = DemoProcessor(models.create_model(opt), max_batch=16, max_wait_ms=2.0)
    result_pil = proc.process_image(image_pil, mask_pil)       # callable from any number of threads
    proc.close()

Everything except the forward itself (``run_batch``) is plain host logic and is unit-tested on the CPU with a fake forward.
"""
import threading
import time
from collections import OrderedDict, deque

import numpy as np


class _Request:
    __slots__ = ("key", "payload", "event", "result", "error", "t_submit")

    def __init__(self, key, payload):
        self.key, self.payload = key, payload
        self.event = threading.Event()
        self.result = self.error = None
        self.t_submit = time.monotonic()


class RequestBatcher:
    """Thread-safe request batching.

    ``run_batch(key, payloads) -> list of results`` (same length and order) is called from ONE worker thread with all the
    pending requests that share ``key`` (at most ``max_batch``). A request is dispatched as soon as ``max_batch`` requests of
    its key are pending or ``max_wait_ms`` after it was submitted, whichever comes first; keys are served oldest request first.
    ``submit`` blocks the calling thread until its result is ready and re-raises the worker's exception for that batch.
    """

    def __init__(self, run_batch, max_batch=16, max_wait_ms=2.0):
        if max_batch < 1:
            raise ValueError("max_batch must be >= 1")
        self.run_batch, self.max_batch, self.max_wait = run_batch, int(max_batch), max_wait_ms / 1e3
        self._cv = threading.Condition()
        self._pending = OrderedDict()          # key -> deque of requests, keys in order of their oldest pending request
        self._closed = False
        self.batches = []                      # (key, size) of every dispatched batch (observability / tests)
        self._worker = threading.Thread(target=self._loop, name="sketchedit-batcher", daemon=True)
        self._worker.start()

    def submit(self, key, payload):
        req = _Request(key, payload)
        with self._cv:
            if self._closed:
                raise RuntimeError("RequestBatcher is closed")
            self._pending.setdefault(key, deque()).append(req)
            self._cv.notify_all()
        req.event.wait()
        if req.error is not None:
            raise req.error
        return req.result

    def close(self):
        with self._cv:
            self._closed = True
            self._cv.notify_all()
        self._worker.join()

    # -- worker
    def _take(self):
        """Under the lock: the next batch to run, or (None, seconds to sleep) / (None, None) when closed and drained."""
        now = time.monotonic()
        best_wait = None
        for key, q in self._pending.items():
            age = now - q[0].t_submit
            if len(q) >= self.max_batch or age >= self.max_wait or self._closed:
                reqs = [q.popleft() for _ in range(min(self.max_batch, len(q)))]
                if not q:
                    del self._pending[key]
                else:
                    self._pending.move_to_end(key)          # the rest of this key queues behind the other keys
                return reqs, None
            w = self.max_wait - age
            best_wait = w if best_wait is None else min(best_wait, w)
        if self._closed and not self._pending:
            return None, None
        return None, (best_wait if best_wait is not None else 3600.0)

    def _loop(self):
        while True:
            with self._cv:
                reqs, wait = self._take()
                while reqs is None:
                    if wait is None:
                        return
                    self._cv.wait(timeout=wait)
                    reqs, wait = self._take()
            key = reqs[0].key
            try:
                results = self.run_batch(key, [r.payload for r in reqs])
                if len(results) != len(reqs):
                    raise RuntimeError("run_batch returned %d results for %d requests" % (len(results), len(reqs)))
                for r, res in zip(reqs, results):
                    r.result = res
            except BaseException as e:      # noqa: BLE001 - delivered to every requester of this batch
                for r in reqs:
                    r.error = e
            self.batches.append((key, len(reqs)))
            for r in reqs:
                r.event.set()


def floor8(n):
    return n // 8 * 8


class DemoProcessor:
    """``process_image`` of the reference demo (demo.py:39-73) on the batched uint8 forward.

    Differences from the reference function, none of them numerical: it returns the PIL result instead of writing
    ``static/results/<name>``, and concurrent calls share forwards. ``precision``: 'bf16' | 'fp32' | 'fp32_direct'.
    """

    def __init__(self, model, precision=None, max_batch=16, max_wait_ms=2.0, resize="host"):
        import torch
        if resize not in ("host", "device"):
            raise ValueError("resize must be 'host' or 'device' (got %r)" % (resize,))
        self._torch = torch
        self.model = model
        self.precision = precision or getattr(model, "precision", "bf16")
        self.resize = resize
        self.engine = model.engine()
        run = self._run_batch_device if resize == "device" else self._run_batch
        self.batcher = RequestBatcher(run, max_batch=max_batch, max_wait_ms=max_wait_ms)

    def close(self):
        self.batcher.close()

    def _forward_u8(self, img, planes):
        """planes: (sketch,) -> the netM forward; (sketch, region) -> the region inpaint (Engine.inpaint_u8). Returns BGR uint8."""
        with self._torch.no_grad():
            if len(planes) == 2:
                return self.engine.inpaint_u8(img, *planes, precision=self.precision)
            return self.engine.inference_u8(img, *planes, precision=self.precision)[0]

    def _run_batch(self, key, payloads):
        torch, dev = self._torch, self.engine.device
        img = torch.from_numpy(np.stack([p[0] for p in payloads])).to(dev, non_blocking=True)           # [B,H,W,3] RGB uint8
        planes = [torch.from_numpy(np.stack([p[k] for p in payloads])).to(dev, non_blocking=True)        # [B,H,W] uint8 (> 0 = stroke,
                  for k in range(1, len(payloads[0]))]                                                  # > 0 = edit here)
        rgb = self._forward_u8(img, planes).cpu().numpy()[..., ::-1]                                    # demo.py keeps RGB (test.py swaps to BGR)
        return [np.ascontiguousarray(rgb[i]) for i in range(len(payloads))]

    def _run_batch_device(self, key, payloads):
        """payloads: (raw RGB image [h,w,3], raw 'L' mask [h',w'][, raw 'L' region [h'',w'']]) of any raw sizes that floor to
        ``key``. One copy in, the resizes of demo.py:45,49,68 (the region's like the mask's) and the forward on the device, one copy
        out."""
        torch, eng = self._torch, self.engine
        B, n = len(payloads), len(payloads[0])
        size = tuple(key[:2])
        arrays = [p[k] for k in range(n) for p in payloads]              # images, then masks, then regions
        offsets = np.concatenate([[0], np.cumsum([a.nbytes for a in arrays])])
        host = torch.empty(int(offsets[-1]), dtype=torch.uint8, pin_memory=eng.device.type == "cuda")
        flat = host.numpy()
        for a, o in zip(arrays, offsets):
            flat[o:o + a.nbytes] = a.reshape(-1)
        raw = host.to(eng.device, non_blocking=True)
        raw_hw = [a.shape[:2] for a in arrays]
        img = eng.resize_u8(raw, [size] * B, src_hw=raw_hw[:B], channels=3, src_offsets=offsets[:B]).view(B, *size, 3)
        planes = [eng.resize_u8(raw, [size] * B, src_hw=raw_hw[k * B:(k + 1) * B], channels=1, src_offsets=offsets[k * B:(k + 1) * B]).view(B, *size)
                  for k in range(1, n)]
        bgr = self._forward_u8(img, planes)
        rgb = eng.resize_u8(bgr, raw_hw[:B], src_hw=[size] * B, channels=3, reverse_channels=True).cpu().numpy()
        ends = np.cumsum([h * w * 3 for h, w in raw_hw[:B]])
        return [rgb[e - h * w * 3:e].reshape(h, w, 3) for e, (h, w) in zip(ends, raw_hw[:B])]

    def process_image(self, img, mask, region=None):
        """img: PIL image; mask: PIL 'L' image of the same size (non-zero = sketch stroke). Returns the edited PIL image at the
        input's size. Sizes are floored to a multiple of 8 for the network exactly like demo.py:43. With resize='device' the
        mask must be mode 'L' (Pillow resizes some other modes with another filter); its size may differ from the image's.

        region: None (netM chooses where to edit) or a PIL 'L' image, non-zero = edit here, resized and binarised exactly like the
        mask. The edit then stays inside it (``Engine.inpaint_u8``); such requests batch apart from plain ones, under
        ``(h, w, "region")``."""
        from PIL import Image
        img = img.convert("RGB")
        w_raw, h_raw = img.size
        h_t, w_t = floor8(h_raw), floor8(w_raw)
        if h_t < 16 or w_t < 16:
            raise ValueError("image smaller than 16x16 (two stride-2 convolutions, 4x4 mask pool, stride-2 patch grid)")
        planes = (mask,) if region is None else (mask, region)
        key = (h_t, w_t) if region is None else (h_t, w_t, "region")
        if self.resize == "device":
            for p in planes:
                if p.mode != "L":
                    raise ValueError("resize='device' needs 'L' masks and regions (got mode %r)" % p.mode)
            return Image.fromarray(self.batcher.submit(key, (np.asarray(img),) + tuple(np.asarray(p) for p in planes)))
        img_t = np.ascontiguousarray(np.array(img.resize((w_t, h_t))), dtype=np.uint8)
        planes_t = tuple(np.ascontiguousarray((np.array(p.resize((w_t, h_t))) > 0).astype(np.uint8) * 255) for p in planes)
        out = self.batcher.submit(key, (img_t,) + planes_t)
        return Image.fromarray(out).resize((w_raw, h_raw))
