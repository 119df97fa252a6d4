"""GPU parity at the sizes BASELINE.json's configs are quoted on (everything else in tests/ uses small shapes):

  config 2   256x256, batch 32, fp32 path, 1e-3 vs the oracle
  config 3   256x256, batch 128, bf16 tensor-core path (the bench shape), 1e-2 vs the fp32 oracle
  config 4   Places-size inputs: 512x512 batch 16 and the reference's own 408-wide x 512-high input (contextual
             attention over L = 3969 / 3150 patches)
  config 5   data-parallel shards + NCCL all-gather == the single-GPU result bit for bit (needs >= 2 GPUs)

plus the module-surface pieces the reference's callers use: mode='visualize' (reference models/editline2_model.py:134-145)
and the whole test.py flow (reference test.py:12-37) on a list file + checkpoints, compared PNG against PNG.

At these sizes every image of a batch must equal the same image run alone BIT FOR BIT (size-independent property: no op
mixes samples, SURVEY.md 8e) and a sample of images is checked against the CPU oracle.
"""
import os

import numpy as np
import pytest
import torch

from oracle import sketchedit_oracle as O
from oracle.golden import Golden
from sketchedit_b200 import synth
from tests.util_parity import engine, maxdiff, weights

pytestmark = pytest.mark.gpu
TOL = {"fp32": 1e-3, "fp32_direct": 1e-3, "bf16": 1e-2}


def _oracle(img, sk, mask_bin=None, chunk=2):
    """Oracle in chunks of `chunk` images (bounds the L x L attention tensors at 512x512)."""
    WM, WG = weights()
    outs = []
    for i in range(0, img.shape[0], chunk):
        mb = None if mask_bin is None else mask_bin[i:i + chunk]
        outs.append(O.inference(WM, WG, img[i:i + chunk], sk[i:i + chunk], mask_bin_override=mb))
    return {k: torch.cat([o[k] for o in outs]) for k in outs[0]}


def _check_batch(prec, B, H, W, seed, sample, singles):
    img, sk = synth.synth_inputs(B, H, W, seed=seed)
    eng = engine()
    comp, mask, ex = eng.inference(img.cuda(), sk.cuda(), precision=prec, want=("mask_bin", "fine"))
    torch.cuda.synchronize()
    # (1) batch independence, bit for bit
    bad = []
    for i in singles:
        c1, m1, _ = eng.inference(img[i:i + 1].cuda(), sk[i:i + 1].cuda(), precision=prec)
        if not (torch.equal(c1[0], comp[i]) and torch.equal(m1[0], mask[i])):
            bad.append((i, float((c1[0] - comp[i]).abs().max()), float((m1[0] - mask[i]).abs().max())))
    assert not bad, "images of the batch that differ from their batch-1 run (index, max|d composed|, max|d mask|): %r" % (bad[:16],)
    # (2) parity of a sample against the oracle (netG compared on OUR binarised mask; threshold flips bounded separately)
    idx = torch.tensor(sample)
    ours_bin = ex["mask_bin"].cpu()[idx]
    free = _oracle(img[idx], sk[idx])
    flipped = ours_bin != free["mask_bin"]
    flips = int(flipped.sum())
    if prec == "fp32_direct":
        assert flips == 0, flips
    elif prec == "fp32":
        # split-half fp16 tensor-core products carry ~22 bits: a pixel may land on the other side of the 0.5 threshold only where
        # the oracle's own soft mask is within fp32 reordering noise of it (any fp32 implementation flips those, cuDNN included)
        margin = (free["mask"] - 0.5).abs()[flipped]
        assert flips <= 2e-5 * ours_bin.numel() and (flips == 0 or float(margin.max()) <= 5e-5), (flips, margin.max() if flips else 0)
    else:
        assert flips <= 0.02 * ours_bin.numel(), flips
    ref = free if flips == 0 else _oracle(img[idx], sk[idx], mask_bin=ours_bin)
    assert maxdiff(mask.cpu()[idx], ref["mask"]) <= TOL[prec]
    assert maxdiff(ex["fine"].cpu()[idx], ref["fine"]) <= TOL[prec], maxdiff(ex["fine"].cpu()[idx], ref["fine"])
    assert maxdiff(comp.cpu()[idx], ref["composed"]) <= TOL[prec], maxdiff(comp.cpu()[idx], ref["composed"])


def test_config3_bf16_batch128_256():
    """The bench shape: 65 536 tiles per 256^2 launch, every ring of the tcgen05 kernels wraps thousands of times."""
    _check_batch("bf16", 128, 256, 256, seed=77, sample=[0, 17, 34, 51, 68, 85, 102, 127], singles=range(128))


def test_config2_fp32_batch32_256():
    _check_batch("fp32", 32, 256, 256, seed=78, sample=[0, 5, 9, 14, 18, 23, 27, 31], singles=[0, 13, 31])


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_config4_places_batch16_512(prec):
    _check_batch(prec, 16, 512, 512, seed=79, sample=[0, 6, 11, 15], singles=[3, 15])


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_config4_places_native_512x408(prec):
    """Non-square Places input (H=512, W=408 like datasets/general_release/images/11.png): L = 63 * 50 = 3150."""
    _check_batch(prec, 1, 512, 408, seed=80, sample=[0], singles=[])


def test_bf16_places_golden(golden_dir):
    """bf16 path on the reference's own 408x512 general-scene input vs outputs of the unmodified reference."""
    g = Golden(os.path.join(golden_dir, "places_11_512x408.npz"))
    image, sketch = g.inputs()
    composed, mask, ex = engine().inference(image.cuda(), sketch.cuda(), precision="bf16", want=("mask_bin",))
    assert g.maxdiff("mask", mask) <= 1e-2
    ours_bin = ex["mask_bin"].cpu()
    ref_bin = g.mask_bin()
    assert int((ours_bin != ref_bin).sum()) <= 0.02 * ours_bin.numel()
    WM, WG = weights()
    ref = O.inference(WM, WG, image, sketch, mask_bin_override=ours_bin)
    assert maxdiff(composed.cpu(), ref["composed"]) <= 1e-2


# ------------------------------------------------------------------------------------------------ module surface
def _model(prec, **over):
    from argparse import Namespace

    import models
    opt = Namespace(gpu_ids=[0], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02,
                    use_cam=True, pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True,
                    model="editline2", precision=prec)
    for k, v in over.items():
        setattr(opt, k, v)
    model = models.create_model(opt)
    model.netM.load_state_dict(synth.synth_state_dict("M"))
    model.netG.load_state_dict(synth.synth_state_dict("G"))
    return model.eval()


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_visualize_contract(prec):
    """mode='visualize' (reference editline2_model.py:134-145): mask = BINARISED mask, maskim = netM image head, coarse,
    fine, composed = soft-mask blend; exactly these five keys."""
    img, sk = synth.synth_inputs(2, 64, 96, seed=31)
    model = _model(prec)
    with torch.no_grad():
        vis = model({"image": img, "mask": sk}, mode="visualize")
        comp_inf, mask_inf = model({"image": img, "mask": sk}, mode="inference")
    assert sorted(vis) == ["coarse", "composed", "fine", "mask", "maskim"]
    assert set(vis["mask"].unique().tolist()) <= {0.0, 1.0}
    assert torch.equal(vis["mask"], (mask_inf > 0.5).float())
    assert torch.equal(vis["composed"], comp_inf)
    WM, WG = weights()
    ref = O.inference(WM, WG, img, sk, mask_bin_override=vis["mask"].cpu())
    assert int((vis["mask"].cpu() != O.inference(WM, WG, img, sk)["mask_bin"]).sum()) <= (0 if prec == "fp32" else 0.02 * sk.numel())
    for ours, key in ((vis["maskim"], "mask_image"), (vis["coarse"], "coarse"), (vis["fine"], "fine"), (vis["composed"], "composed")):
        assert maxdiff(ours.cpu(), ref[key]) <= TOL[prec], (key, maxdiff(ours.cpu(), ref[key]))
    # composed blends with the SOFT mask (:138), not the binarised one
    soft = vis["fine"] * mask_inf + img.cuda() * (1 - mask_inf)
    assert maxdiff(vis["composed"].cpu(), soft.cpu()) <= 1e-6


def test_netG_guide_none():
    """guide=None -> all-ones sketch channel (reference editline_g.py:127-130), through the C ABI."""
    _, WG = weights()
    img, sk = synth.synth_inputs(1, 64, 64, seed=33)
    mask = torch.zeros(1, 1, 64, 64)
    mask[:, :, 20:44, 12:50] = 1
    s1, s2 = engine().netG(img.cuda(), img.cuda(), mask.cuda(), mask.cuda(), None, precision="fp32")
    r1, r2 = O.netG_forward(WG, img, img, mask, mask, None)
    assert maxdiff(s1.cpu(), r1) <= 1e-3 and maxdiff(s2.cpu(), r2) <= 1e-3


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_test_py_end_to_end(prec, tmp_path):
    """The reference's entry point (test.py:12-37 with the flags of test_celeb.sh) on a list file, PNG inputs and
    `<checkpoints_dir>/<name>/latest_net_{G,M}.pth`: the PNGs it writes are (a) byte-for-byte the oracle's uint8 conversion
    (test.py:25-35: truncate, CHW->HWC, RGB->BGR) of this path's own float outputs and (b), on the fp32 path, within one
    grey level of the CPU oracle's PNG everywhere (the float outputs agree to ~1e-6; truncation can split a tie)."""
    import cv2
    from PIL import Image

    import test as test_entry
    from tests.test_host_surface import _script_args
    idir, mdir, odir, omdir, cdir = (tmp_path / n for n in ("images", "edges", "out", "out_mask", "ckpt"))
    idir.mkdir(); mdir.mkdir(); (cdir / "celeb").mkdir(parents=True)
    WM, WG = weights()
    torch.save(WM, cdir / "celeb" / "latest_net_M.pth")
    torch.save({"module." + k: v for k, v in WG.items()}, cdir / "celeb" / "latest_net_G.pth")   # DataParallel prefix is stripped
    names, tensors = [], {}
    for j, (H, W) in enumerate(((64, 64), (64, 64), (96, 64))):
        img, sk = synth.synth_inputs(1, H, W, seed=40 + j)
        u8 = ((img[0].permute(1, 2, 0) + 1) / 2 * 255).round().clamp(0, 255).to(torch.uint8).numpy()
        e8 = (sk[0, 0] * 255).to(torch.uint8).numpy()
        n = "im_%02d" % j
        Image.fromarray(u8).save(idir / (n + ".png"))
        Image.fromarray(e8).save(mdir / (n + ".png"))
        names.append(n)
        tensors[n] = (torch.from_numpy(u8).permute(2, 0, 1).float().div(255).sub(0.5).div(0.5)[None], (torch.from_numpy(e8).float().div(255) > 0).float()[None, None])
    (tmp_path / "list.txt").write_text("".join(n + ".png\n" for n in names))
    argv = _script_args("test_celeb.sh") + ["--image_dirs", str(idir), "--mask_dirs", str(mdir), "--image_lists", str(tmp_path / "list.txt"),
                                            "--output_dir", str(odir), "--output_mask_dir", str(omdir), "--checkpoints_dir", str(cdir),
                                            "--precision", prec, "--nThreads", "0"]
    test_entry.main(argv)
    eng = engine()
    for n in names:
        got = cv2.imread(str(odir / (n + ".png")), cv2.IMREAD_COLOR)          # BGR, HWC
        got_m = cv2.imread(str(omdir / (n + ".png")), cv2.IMREAD_GRAYSCALE)
        image, sketch = tensors[n]
        comp, mask, ex = eng.inference(image.cuda(), sketch.cuda(), precision=prec, want=("mask_bin",))
        g, m = O.to_uint8_outputs(comp.cpu(), mask.cpu())
        assert np.array_equal(got, g[0].transpose(1, 2, 0)[..., ::-1]), n
        assert np.array_equal(got_m, m[0]), n
        if prec == "fp32":
            ref = O.inference(WM, WG, image, sketch)
            flipped = ex["mask_bin"].cpu() != ref["mask_bin"]
            if bool(flipped.any()):   # a soft-mask value within fp32 noise of the 0.5 threshold (see _check_batch): compare netG on OUR mask
                assert int(flipped.sum()) <= 2 and float((ref["mask"] - 0.5).abs()[flipped].max()) <= 5e-5
                ref = O.inference(WM, WG, image, sketch, mask_bin_override=ex["mask_bin"].cpu())
            rg, rm = O.to_uint8_outputs(ref["composed"], ref["mask"])
            d = np.abs(got.astype(int) - rg[0].transpose(1, 2, 0)[..., ::-1].astype(int))
            assert d.max() <= 1 and (d != 0).mean() <= 2e-3, (d.max(), (d != 0).mean())   # truncation ties: |err| ~1e-5 of 1/127.5 per level
            assert np.abs(got_m.astype(int) - rm[0].astype(int)).max() <= 1


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_uint8_codecs_on_device(prec):
    """Engine.inference_u8 (input codec: x/255 -> (x-0.5)/0.5, sketch > 0; output codec fused into the heads) is byte for byte
    the float forward on host-decoded inputs followed by the oracle's test.py conversion."""
    rs = np.random.RandomState(5)
    img_u8 = torch.from_numpy(rs.randint(0, 256, (2, 64, 96, 3), dtype=np.uint8))
    _, sk = synth.synth_inputs(2, 64, 96, seed=44)
    sk_u8 = (sk[:, 0] * 255).to(torch.uint8)
    sk_u8[0, 10:14, 5:40] = 7          # any non-zero value is sketch (reference: ToTensor then > 0)
    image = img_u8.permute(0, 3, 1, 2).float().div(255).sub(0.5).div(0.5)        # reference data/testimage_dataset.py:89-103
    sketch = (sk_u8.float().div(255)[:, None] > 0).float()
    eng = engine()
    bgr, mk = eng.inference_u8(img_u8.cuda(), sk_u8.cuda(), precision=prec)
    comp, mask, _ = eng.inference(image.cuda(), sketch.cuda(), precision=prec)
    g, m = O.to_uint8_outputs(comp.cpu(), mask.cpu())
    assert np.array_equal(bgr.cpu().numpy(), g.transpose(0, 2, 3, 1)[..., ::-1])
    assert np.array_equal(mk.cpu().numpy(), m)


def test_uint8_stream_matches_blocking_calls():
    model = _model("bf16")
    rs = np.random.RandomState(6)
    batches = []
    for i, b in enumerate((2, 2, 2, 1)):
        _, sk = synth.synth_inputs(b, 64, 64, seed=70 + i)
        batches.append({"image_u8": torch.from_numpy(rs.randint(0, 256, (b, 64, 64, 3), dtype=np.uint8)).pin_memory(),
                        "mask_u8": (sk[:, 0] * 255).to(torch.uint8).pin_memory(), "tag": i})
    eng = model.engine()
    with torch.no_grad():
        want = [tuple(t.cpu() for t in eng.inference_u8(d["image_u8"].cuda(), d["mask_u8"].cuda(), precision="bf16")) for d in batches]
        got = [(a.clone(), b.clone(), d["tag"]) for a, b, d in model.inference_stream(iter(batches), uint8=True, with_data=True)]
    assert [t for _, _, t in got] == [0, 1, 2, 3]
    for (ga, gb, _), (wa, wb) in zip(got, want):
        assert torch.equal(ga, wa) and torch.equal(gb, wb)


def test_stream_ring_keeps_depth_plus_one_results():
    """inference_stream's pinned ring (depth + 2 buffers, strict round robin): the newest `depth + 1` results stay intact
    -- held WITHOUT cloning (the copy of batch i + depth - 1 is in flight when result i is drawn)."""
    model = _model("bf16")
    batches = []
    for i in range(7):
        img, sk = synth.synth_inputs(1, 64, 64, seed=60 + i)
        batches.append({"image": img.pin_memory(), "mask": sk.pin_memory()})
    with torch.no_grad():
        want = [tuple(t.cpu() for t in model(d, mode="inference")) for d in batches]
        held = []
        for k, (c, m) in enumerate(model.inference_stream(iter(batches), depth=2)):
            held.append((k, c, m))
            held = held[-3:]                       # depth + 1 = 3 newest results
            torch.cuda.synchronize()               # every copy issued so far has landed: nothing may have overwritten them
            for kk, cc, mm in held:
                assert torch.equal(cc, want[kk][0]) and torch.equal(mm, want[kk][1]), (k, kk)


# ------------------------------------------------------------------------------------------------ config 5
def _dp_worker(rank, world, port, B, ret):
    import torch.distributed as dist

    from sketchedit_b200 import parallel
    from sketchedit_b200.engine import Engine
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    eng = Engine.from_state_dicts(synth.synth_state_dict("M"), synth.synth_state_dict("G"))
    img, sk = synth.synth_inputs(world * B, 64, 64, seed=90)
    lo, hi = parallel.shard_bounds(world * B, world, rank)
    g = parallel.OutputGather(B, 64, 64, torch.device("cuda", rank))
    full = None
    for _ in range(3):                              # several rounds: both ring buffers, in-flight collectives
        slot = g.next_slot()
        eng.inference_packed(img[lo:hi].cuda(), sk[lo:hi].cuda(), precision="bf16", out=slot)
        g.launch()
        full = g.wait()
    torch.cuda.synchronize()
    if rank == 0:
        comp, mask, _ = eng.inference(img.cuda(), sk.cuda(), precision="bf16")
        ret["ok"] = bool(torch.equal(full[:, :3], comp) and torch.equal(full[:, 3:4], mask))
    dist.barrier()
    dist.destroy_process_group()


def test_config5_gathered_equals_single_gpu():
    """Batch shards on 2 GPUs + the in-place NCCL all-gather of the packed outputs == one GPU computing the whole batch,
    bit for bit (config 5)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    from tests.test_parallel_gloo import _free_port
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dp_worker, args=(2, _free_port(), 3, ret), nprocs=2, join=True)
    assert ret.get("ok") is True
