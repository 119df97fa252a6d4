"""Format of the reference-generated vectors under tests/golden/ (written by oracle/make_golden.py).

Each .npz keeps in full what a forward needs and what must agree exactly: the inputs, the flags and the reference's
binarised mask (``mask_bin``, bit-packed). Every float output and tap ``<key>`` is kept as a fixed, seeded sample of its
elements, stored with their flat indices (``<key>:idx``), the full array's shape (``<key>:shape``) and its largest
magnitude (``<key>:absmax``): full-resolution float outputs would not fit in files under 1 MB.
"""
import numpy as np
import torch

SAMPLE_ELEMENTS = 80000     # float elements kept per file, split evenly over its outputs and taps


def save(path, inputs, outputs, flags, seed=0):
    """inputs: {name: array} stored whole; outputs: {name: float array}, "mask" among them, sampled."""
    rs = np.random.RandomState(seed)
    cap = SAMPLE_ELEMENTS // len(outputs)
    out = dict(inputs)
    out["mask_bin"] = np.packbits(np.asarray(outputs["mask"]).ravel() > 0.5)
    for key, v in outputs.items():
        v = np.asarray(v, np.float32)
        idx = np.arange(v.size) if v.size <= cap else np.sort(rs.choice(v.size, cap, replace=False))
        out[key] = v.ravel()[idx]
        out[key + ":idx"] = idx.astype(np.int32)
        out[key + ":shape"] = np.array(v.shape, np.int64)
        out[key + ":absmax"] = np.float32(np.abs(v).max())
    out["flags"] = np.array(repr(sorted(flags.items())))
    np.savez_compressed(path, **out)


class Golden:
    def __init__(self, path):
        self.z = np.load(path)
        self.flags = dict(eval(str(self.z["flags"])))
        self.keys = [k for k in self.z.files if k + ":idx" in self.z.files]

    def __contains__(self, key):
        return key in self.keys

    def inputs(self):
        """(image [B,3,H,W] in [-1, 1], sketch [B,1,H,W] in {0, 1}); uint8 pairs get the reference's dataset preprocessing
        (data/testimage_dataset.py)."""
        z = self.z
        if "image" in z:
            return torch.from_numpy(z["image"]), torch.from_numpy(z["sketch"])
        image = torch.from_numpy(z["image_u8"]).permute(2, 0, 1).float().div(255).sub(0.5).div(0.5)[None]
        sketch = (torch.from_numpy(z["sketch_u8"]).float().div(255) > 0).float()[None, None]
        return image, sketch

    def shape(self, key):
        return tuple(int(s) for s in self.z[key + ":shape"])

    def mask_bin(self):
        """The reference's mask > 0.5, every pixel, as a float 0/1 tensor."""
        shape = self.shape("mask")
        bits = np.unpackbits(self.z["mask_bin"], count=int(np.prod(shape)))
        return torch.from_numpy(bits.astype(np.float32).reshape(shape))

    def absmax(self, key):
        return float(self.z[key + ":absmax"])

    def maxdiff(self, key, ours):
        """max |ours - reference| over the stored elements of `key`; `ours` is the whole array."""
        ours = torch.as_tensor(ours).detach().cpu()
        assert tuple(ours.shape) == self.shape(key), (key, tuple(ours.shape), self.shape(key))
        got = ours.reshape(-1)[torch.from_numpy(self.z[key + ":idx"]).long()]
        return float((got.float() - torch.from_numpy(self.z[key])).abs().max())
