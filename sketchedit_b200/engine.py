"""Torch-tensor front end of the C ABI: owns an ``se_model`` (packed weights on the GPU) and
exposes the reference's call surface for the generator forward pass with CUDA tensors in and out.

    eng = Engine.from_state_dicts(sd_M, sd_G, use_cam=True, pool_type="max", joint_train_inp=True)
    composed, mask = eng.inference(image_cuda, sketch_cuda, precision="bf16")

PyTorch is plumbing here (device memory + current stream); all compute is in libsketchedit_b200.so.
"""
import ctypes
from itertools import accumulate

import numpy as np
import torch

from . import _lib
from .arch import NET_LAYERS, layer_map, out_channels_after_gate


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk_in(t, shape_tail=None, name="tensor"):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32):
        raise _lib.SketchEditB200Error("%s must be a CUDA float32 tensor (got %r)" % (name, getattr(t, "device", type(t))))
    return t.contiguous()


def _chk_out(t, shape, name):
    """Caller-owned output: the kernels write through its pointer, so a silent .contiguous() copy is not an option."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise _lib.SketchEditB200Error("%s must be a contiguous CUDA float32 tensor" % name)
    if tuple(t.shape) != tuple(shape):
        raise _lib.SketchEditB200Error("%s must have shape %r (got %r)" % (name, tuple(shape), tuple(t.shape)))
    return t


def _f32(*shape, like):
    return torch.empty(*shape, device=like.device, dtype=torch.float32)


def _chk_u8(t, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous()):
        raise _lib.SketchEditB200Error("%s must be a contiguous CUDA uint8 tensor" % name)
    return t


def resize_u8(src, dst_hw, src_hw=None, channels=None, src_offsets=None, out=None, out_offsets=None, reverse_channels=False):
    """Pillow's ``Image.resize((w, h))`` with its default filter (BICUBIC) on the device, bit for bit (se_resize_u8): a ragged
    batch of uint8 HWC images, image i to size ``dst_hw[i] = (h, w)``, one launch per pass. Uses no model.

    * ``src`` a list of CUDA uint8 tensors [H,W,C] (C = 1 or 3) or [H,W]: returns a list of tensors [h,w,C] (or [h,w]), views of
      one new buffer.
    * ``src`` a packed CUDA uint8 buffer with ``src_hw`` (one (H, W) per image) and ``channels``: the images lie back to back, or at
      byte offsets ``src_offsets``. Returns the flat output buffer with the results back to back, or writes them into ``out``
      at byte offsets ``out_offsets`` and returns ``out``.

    ``reverse_channels`` writes the channels reversed (RGB <-> BGR)."""
    listed = isinstance(src, (list, tuple))
    if listed:
        if not src:
            return []
        for i, t in enumerate(src):
            _chk_u8(t, "src[%d]" % i)
            if t.dim() not in (2, 3) or t.device != src[0].device:
                raise _lib.SketchEditB200Error("src[%d] must be [H,W] or [H,W,C] on %s" % (i, src[0].device))
        shapes = {t.shape[2:] for t in src}
        if len(shapes) != 1:
            raise _lib.SketchEditB200Error("all images of a batch need the same channel count")
        channels = src[0].shape[2] if src[0].dim() == 3 else 1
        src_hw = [tuple(t.shape[:2]) for t in src]
        base = min(t.data_ptr() for t in src)
        src_offsets = [t.data_ptr() - base for t in src]
        device = src[0].device
    else:
        _chk_u8(src, "src")
        if src_hw is None or channels is None:
            raise _lib.SketchEditB200Error("a packed src needs src_hw and channels")
        base, device = src.data_ptr(), src.device
    B, C = len(src_hw), int(channels)
    if len(dst_hw) != B:
        raise _lib.SketchEditB200Error("dst_hw has %d sizes for %d images" % (len(dst_hw), B))
    if min(min(hw) for hw in list(src_hw) + list(dst_hw)) < 1:
        raise _lib.SketchEditB200Error("image sizes must be positive")
    src_n = [int(h) * int(w) * C for h, w in src_hw]
    dst_n = [int(h) * int(w) * C for h, w in dst_hw]
    if src_offsets is None:
        src_offsets = [0] + list(accumulate(src_n))[:-1]
    if not listed and any(o < 0 or o + n > src.numel() for o, n in zip(src_offsets, src_n)):
        raise _lib.SketchEditB200Error("an image lies outside src")
    if out is None:
        if out_offsets is not None:
            raise _lib.SketchEditB200Error("out_offsets needs out")
        out = torch.empty(sum(dst_n), device=device, dtype=torch.uint8)
    elif _chk_u8(out, "out").device != device:
        raise _lib.SketchEditB200Error("out must be on %s" % device)
    if out_offsets is None:
        out_offsets = [0] + list(accumulate(dst_n))[:-1]
    if any(o < 0 or o + n > out.numel() for o, n in zip(out_offsets, dst_n)):
        raise _lib.SketchEditB200Error("an image lies outside out")
    i64 = lambda v: np.ascontiguousarray(v, dtype=np.int64)
    i32 = lambda v: np.ascontiguousarray(np.asarray(v, dtype=np.int64).reshape(B, 2), dtype=np.int32)
    so, shw, do, dhw = i64(src_offsets), i32(src_hw), i64(out_offsets), i32(dst_hw)
    with torch.cuda.device(device):
        _lib.check(_lib.load().se_resize_u8(ctypes.c_void_p(base), so.ctypes.data, shw.ctypes.data, B, C, _ptr(out), do.ctypes.data,
                                            dhw.ctypes.data, _lib.RESIZE_REVERSE_CHANNELS if reverse_channels else 0, _stream()))
    if not listed:
        return out
    return [out[o:o + n].view(h, w, C) if src[i].dim() == 3 else out[o:o + n].view(h, w)
            for i, (o, n, (h, w)) in enumerate(zip(out_offsets, dst_n, dst_hw))]


class Engine:
    def __init__(self):
        self.lib = _lib.load()
        h = ctypes.c_void_p()
        _lib.check(self.lib.se_model_create(ctypes.byref(h)))
        self.h = h
        self.finalized = False

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.se_model_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -------------------------------------------------------------------------------- weights
    def set_layer(self, net, name, weight, bias):
        w = weight.detach().to("cpu", torch.float32).contiguous()
        b = bias.detach().to("cpu", torch.float32).contiguous()
        cout, cin, k, k2 = w.shape
        assert k == k2
        _lib.check(self.lib.se_model_set_layer(self.h, net.encode(), name.encode(), ctypes.c_void_p(w.data_ptr()),
                                               ctypes.c_void_p(b.data_ptr()), cout, cin, k))

    def load_state_dict(self, net, sd):
        """sd: reference-format state_dict ('<layer>.weight', '<layer>.bias'; optional 'module.' prefix,
        stripped like reference util/util.py:221-222). Strict: every layer of the net must be present."""
        sd = {(k[7:] if k.startswith("module.") else k): v for k, v in sd.items()}
        expect = set()
        for l in NET_LAYERS[net]:
            expect.add(l.name + ".weight")
            expect.add(l.name + ".bias")
        missing, extra = expect - set(sd), set(sd) - expect
        if missing or extra:
            raise KeyError("state_dict mismatch for net%s: missing %s unexpected %s" % (net, sorted(missing), sorted(extra)))
        for l in NET_LAYERS[net]:
            self.set_layer(net, l.name, sd[l.name + ".weight"], sd[l.name + ".bias"])

    def set_options(self, use_cam=True, pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True):
        if pool_type not in ("max", "avg"):
            raise NotImplementedError(pool_type)          # reference editline_g.py:164-165
        for key, val in (("use_cam", use_cam), ("pool_avg", pool_type == "avg"), ("no_mask_cc", no_mask_cc),
                         ("no_mask_coarse", no_mask_coarse), ("joint_train_inp", joint_train_inp)):
            _lib.check(self.lib.se_model_set_option(self.h, _lib.OPT[key], int(bool(val))))

    def finalize(self):
        if not torch.cuda.is_available():
            raise _lib.SketchEditB200Error("sketchedit_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        _lib.check(self.lib.se_model_finalize(self.h))
        self.finalized = True
        self.device = torch.device("cuda", torch.cuda.current_device())   # weights + workspace live here

    def _on_device(self, *tensors):
        for t in tensors:
            if t is not None and t.device != self.device:
                raise _lib.SketchEditB200Error("tensor on %s but this engine was finalized on %s" % (t.device, self.device))

    @classmethod
    def from_state_dicts(cls, sd_M, sd_G, **options):
        e = cls()
        if sd_M is not None:
            e.load_state_dict("M", sd_M)
        if sd_G is not None:
            e.load_state_dict("G", sd_G)
        e.set_options(**options)
        e.finalize()
        return e

    # -------------------------------------------------------------------------------- forward
    def inference(self, image, sketch, precision="bf16", want=(), mask_bin=None, out=None):
        """EditLine2Model.forward(mode='inference'): returns (composed, mask) and, in a dict, any of
        want = ('coarse', 'fine', 'mask_image', 'mask_bin'). ``out=(composed, mask)`` writes into caller-owned
        fp32 CUDA tensors of shape [B,3,H,W] / [B,1,H,W] instead of allocating (pipelined callers)."""
        image = _chk_in(image, name="image")
        sketch = _chk_in(sketch, name="sketch")
        B, _, H, W = image.shape
        new = lambda c: _f32(B, c, H, W, like=image)
        if out is not None:
            composed, mask = _chk_out(out[0], (B, 3, H, W), "out[0]"), _chk_out(out[1], (B, 1, H, W), "out[1]")
        else:
            composed, mask = new(3), new(1)
        extra = {k: new(1 if k == "mask_bin" else 3) for k in want}
        mb_in = _chk_in(mask_bin, name="mask_bin") if mask_bin is not None else None
        self._on_device(image, sketch, composed, mask, mb_in)
        _lib.check(self.lib.se_forward_inference(
            self.h, _ptr(image), _ptr(sketch), B, H, W, _lib.PREC[precision], _ptr(composed), _ptr(mask),
            _ptr(extra.get("coarse")), _ptr(extra.get("fine")), _ptr(extra.get("mask_image")), _ptr(mb_in),
            _ptr(extra.get("mask_bin")), _stream()))
        return composed, mask, extra

    def inference_packed(self, image, sketch, precision="bf16", out=None):
        """Same forward, ONE packed output [B,4,H,W] (channels 0-2 composed, channel 3 the soft mask) = the layout of the
        data-parallel output all-gather: ``out`` may be this rank's slice of the gather buffer (parallel.OutputGather)."""
        image = _chk_in(image, name="image")
        sketch = _chk_in(sketch, name="sketch")
        B, _, H, W = image.shape
        packed = _f32(B, 4, H, W, like=image) if out is None else _chk_out(out, (B, 4, H, W), "out")
        self._on_device(image, sketch, packed)
        _lib.check(self.lib.se_forward_inference_packed(self.h, _ptr(image), _ptr(sketch), B, H, W, _lib.PREC[precision], _ptr(packed),
                                                        _stream()))
        return packed

    def inference_u8(self, image_u8, sketch_u8, precision="bf16", out=None):
        """Forward with the reference's host-side codecs on the device: image_u8 [B,H,W,3] RGB uint8 and sketch_u8 [B,H,W]
        uint8 (reference data/testimage_dataset.py:89-103 up to ToTensor) -> (bgr_u8 [B,H,W,3], mask_u8 [B,H,W]) exactly as
        test.py:25-35 writes them. ``out=(bgr, mask)`` writes into caller-owned uint8 CUDA tensors."""
        for t, nm in ((image_u8, "image_u8"), (sketch_u8, "sketch_u8")):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous()):
                raise _lib.SketchEditB200Error("%s must be a contiguous CUDA uint8 tensor" % nm)
        B, H, W, C = image_u8.shape
        if C != 3 or tuple(sketch_u8.shape) != (B, H, W):
            raise _lib.SketchEditB200Error("image_u8 must be [B,H,W,3] and sketch_u8 [B,H,W]")
        if out is None:
            bgr = torch.empty(B, H, W, 3, device=image_u8.device, dtype=torch.uint8)
            mk = torch.empty(B, H, W, device=image_u8.device, dtype=torch.uint8)
        else:
            bgr, mk = out
            for t, shp in ((bgr, (B, H, W, 3)), (mk, (B, H, W))):
                if not (t.is_cuda and t.dtype == torch.uint8 and t.is_contiguous() and tuple(t.shape) == shp):
                    raise _lib.SketchEditB200Error("out tensors must be contiguous CUDA uint8 [B,H,W,3] and [B,H,W]")
        self._on_device(image_u8, sketch_u8, bgr, mk)
        _lib.check(self.lib.se_forward_inference_u8(self.h, _ptr(image_u8), _ptr(sketch_u8), B, H, W, _lib.PREC[precision], _ptr(bgr), _ptr(mk),
                                                    _stream()))
        return bgr, mk

    def inpaint(self, image, sketch, region, precision="bf16", want=(), out=None):
        """Edit a region the caller chooses, without netM: ``coarse, fine = netG(image, image, region, region, sketch * region)``
        and ``composed = fine * region + image * (1 - region)``, which equals ``image`` wherever region is 0. image [B,3,H,W] in
        [-1,1], sketch and region [B,1,H,W] (region 1 = edit here). Returns (composed, dict of ``want`` among ('coarse', 'fine'));
        ``out`` is a caller-owned fp32 CUDA tensor [B,3,H,W] for composed."""
        image = _chk_in(image, name="image")
        sketch = _chk_in(sketch, name="sketch")
        region = _chk_in(region, name="region")
        B, _, H, W = image.shape
        for t, nm in ((sketch, "sketch"), (region, "region")):
            if tuple(t.shape) != (B, 1, H, W):
                raise _lib.SketchEditB200Error("%s must have shape %r (got %r)" % (nm, (B, 1, H, W), tuple(t.shape)))
        if set(want) - {"coarse", "fine"}:
            raise _lib.SketchEditB200Error("want may hold 'coarse' and 'fine' (got %r)" % (tuple(want),))
        composed = _f32(B, 3, H, W, like=image) if out is None else _chk_out(out, (B, 3, H, W), "out")
        extra = {k: _f32(B, 3, H, W, like=image) for k in want}
        self._on_device(image, sketch, region, composed)
        _lib.check(self.lib.se_forward_inpaint(self.h, _ptr(image), _ptr(sketch), _ptr(region), B, H, W, _lib.PREC[precision], _ptr(composed),
                                               _ptr(extra.get("coarse")), _ptr(extra.get("fine")), _stream()))
        return composed, extra

    def inpaint_u8(self, image_u8, sketch_u8, region_u8, precision="bf16", out=None):
        """``inpaint`` with the codecs of ``inference_u8``: image_u8 [B,H,W,3] RGB, sketch_u8 and region_u8 [B,H,W] uint8 (non-zero =
        stroke / edit here) -> bgr_u8 [B,H,W,3] as test.py:25-35 writes images. ``out`` is a caller-owned uint8 CUDA tensor."""
        for t, nm in ((image_u8, "image_u8"), (sketch_u8, "sketch_u8"), (region_u8, "region_u8")):
            _chk_u8(t, nm)
        B, H, W, C = image_u8.shape
        if C != 3 or tuple(sketch_u8.shape) != (B, H, W) or tuple(region_u8.shape) != (B, H, W):
            raise _lib.SketchEditB200Error("image_u8 must be [B,H,W,3], sketch_u8 and region_u8 [B,H,W]")
        if out is None:
            bgr = torch.empty(B, H, W, 3, device=image_u8.device, dtype=torch.uint8)
        elif tuple(_chk_u8(out, "out").shape) != (B, H, W, 3):
            raise _lib.SketchEditB200Error("out must be a contiguous CUDA uint8 [B,H,W,3] tensor")
        else:
            bgr = out
        self._on_device(image_u8, sketch_u8, region_u8, bgr)
        _lib.check(self.lib.se_forward_inpaint_u8(self.h, _ptr(image_u8), _ptr(sketch_u8), _ptr(region_u8), B, H, W, _lib.PREC[precision],
                                                  _ptr(bgr), _stream()))
        return bgr

    # the model-less device resize, next to the forward it brackets in serving (and replaceable there by a test double)
    resize_u8 = staticmethod(resize_u8)

    def netM(self, x, guide, precision="bf16", want_image=True):
        x, guide = _chk_in(x), _chk_in(guide)
        B, _, H, W = x.shape
        self._on_device(x, guide)
        mask1 = _f32(B, 1, H, W, like=x)
        st1 = _f32(B, 3, H, W, like=x) if want_image else None
        _lib.check(self.lib.se_netM_forward(self.h, _ptr(x), _ptr(guide), B, H, W, _lib.PREC[precision], _ptr(mask1), _ptr(st1),
                                            _stream()))
        return mask1, st1

    def netG(self, x, x2, mask, mask2, guide, precision="bf16"):
        x, x2, mask, mask2 = _chk_in(x), _chk_in(x2), _chk_in(mask), _chk_in(mask2)
        guide = _chk_in(guide) if guide is not None else None
        B, _, H, W = x.shape
        self._on_device(x, x2, mask, mask2, guide)
        s1 = _f32(B, 3, H, W, like=x)
        s2 = _f32(B, 3, H, W, like=x)
        _lib.check(self.lib.se_netG_forward(self.h, _ptr(x), _ptr(x2), _ptr(mask), _ptr(mask2), _ptr(guide), B, H, W,
                                            _lib.PREC[precision], _ptr(s1), _ptr(s2), _stream()))
        return s1, s2

    def gated_conv(self, net, name, x, precision="bf16"):
        x = _chk_in(x)
        spec = layer_map(net)[name]
        B, cin, H, W = x.shape
        if cin != spec.cin:
            raise _lib.SketchEditB200Error("%s expects %d input channels, got %d" % (name, spec.cin, cin))
        if spec.kind == "deconv":
            Ho, Wo = 2 * H, 2 * W
        else:
            Ho, Wo = (H + spec.stride - 1) // spec.stride, (W + spec.stride - 1) // spec.stride
        self._on_device(x)
        y = _f32(B, out_channels_after_gate(spec), Ho, Wo, like=x)
        _lib.check(self.lib.se_gated_conv_forward(self.h, net.encode(), name.encode(), _ptr(x), B, H, W, _lib.PREC[precision],
                                                  _ptr(y), _stream()))
        return y

    def launches(self):
        return int(self.lib.se_last_launch_count())

    def workspace_bytes(self):
        return int(self.lib.se_workspace_bytes(self.h))


def contextual_attention(feat, mask_s, precision="bf16", want_attn=False):
    """cam_2(cam_1(f, f, mask_s), f, mask_s, {})[0] of netG (reference editline_g.py:203-207)."""
    lib = _lib.load()
    feat, mask_s = _chk_in(feat), _chk_in(mask_s)
    B, C, h, w = feat.shape
    out = _f32(*feat.shape, like=feat)
    attn = None
    if want_attn:
        hs, ws = (h - 4) // 2 + 1, (w - 4) // 2 + 1
        attn = _f32(B, hs * ws, hs * ws, like=feat)
    _lib.check(lib.se_contextual_attention_forward(_ptr(feat), _ptr(mask_s), B, C, h, w, _lib.PREC[precision], _ptr(out), _ptr(attn),
                                                   _stream()))
    return (out, attn) if want_attn else out


def outputs_to_uint8(composed, mask):
    """test.py:25-27 on device -> (uint8 [B,H,W,3] BGR, uint8 [B,H,W])."""
    lib = _lib.load()
    composed, mask = _chk_in(composed), _chk_in(mask)
    B, _, H, W = composed.shape
    bgr = torch.empty(B, H, W, 3, device=composed.device, dtype=torch.uint8)
    mk = torch.empty(B, H, W, device=composed.device, dtype=torch.uint8)
    _lib.check(lib.se_outputs_to_uint8(_ptr(composed), _ptr(mask), B, H, W, _ptr(bgr), _ptr(mk), _stream()))
    return bgr, mk
