"""Pin the CPU oracle against outputs of the UNMODIFIED reference (tests/golden/*.npz, made by oracle/make_golden.py
from the original project; format: oracle/golden.py)."""
import glob
import os

import pytest
import torch

from oracle import sketchedit_oracle as O
from oracle.golden import Golden
from sketchedit_b200 import synth

TOL = 2e-5   # fp32 vs fp32, different op order (attention form vs grouped conv)


@pytest.fixture(scope="module")
def weights():
    return synth.synth_state_dict("M"), synth.synth_state_dict("G")


@pytest.mark.parametrize("name", sorted(os.path.basename(p)[:-4] for p in
                                        glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))))
def test_oracle_matches_reference(name, weights, golden_dir):
    WM, WG = weights
    g = Golden(os.path.join(golden_dir, name + ".npz"))
    image, sketch = g.inputs()
    taps = {}
    r = O.inference(WM, WG, image, sketch, taps=taps, **g.flags)
    # the binarised mask must agree exactly (otherwise nothing downstream is comparable)
    assert int((g.mask_bin() != (r["mask_bin"] > 0.5).float()).sum()) == 0
    for key in ("composed", "mask", "coarse", "fine"):
        if key in g:
            d = g.maxdiff(key, r[key])
            assert d <= TOL, (name, key, d)
    for key in g.keys:
        if key.startswith("tap:"):
            d = g.maxdiff(key, taps[key[4:]])
            scale = max(1.0, g.absmax(key))
            assert d <= TOL * scale * 4, (name, key, d)


def test_uint8_conversion_truncates():
    """test.py:25-27: (x+1)/2*255 -> astype(uint8) truncates; mask*255 likewise."""
    comp = torch.tensor([[[[-1.0, 0.0, 0.999, 1.0]]]]).expand(1, 3, 1, 4)
    mask = torch.tensor([[[[0.0, 0.5, 0.999, 1.0]]]])
    g, m = O.to_uint8_outputs(comp, mask)
    assert g[0, 0, 0].tolist() == [0, 127, 254, 255]
    assert m[0, 0].tolist() == [0, 127, 254, 255]
