"""CPU arm of bench.py: times the UNMODIFIED reference (zengxianyu/sketchedit) on the host cores.

Runs in its own process because the reference's top-level packages are called ``models`` / ``util`` like this
repo's mirrors: here ``baseline/_ref`` (a verbatim, git-ignored copy of the reference's ``models/`` and ``util/``
python files made by ``__graft_entry__.build()`` from /root/reference; it ships to the GPU box with the snapshot)
comes first on sys.path. The model is the reference's own ``EditLine2Model`` built the way
``oracle/make_golden.py`` builds it (``isSkip`` escape hatch, reference models/editline2_model.py:195, then a strict
``load_state_dict`` of the seeded synthetic checkpoints) and the timed call is the reference's public entry point
``model(data, mode='inference')`` (reference models/editline2_model.py:107-133) with ``gt``/``edgegt`` supplied as its
CPU branch needs (:225-242).

    python baseline/ref_runner.py --size 256 --batch 4 --steps 3 --warmup 1 [--threads T] [--face]

Prints one JSON object: {"ok", "kind": "reference", "images_per_s", "s_per_step", "threads", "cores", "batch", "size",
"face_b1_s" (config 1: the reference's 256x256 face 602 + sketch at batch 1, when --face)}.
"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.path.join(HERE, "_ref")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--threads", type=int, default=0, help="0 = calibrate over 8..cpu_count")
    ap.add_argument("--face", action="store_true")
    args = ap.parse_args()
    if not os.path.isfile(os.path.join(REF, "models", "editline2_model.py")):
        print(json.dumps({"ok": False, "why": "baseline/_ref is empty (run __graft_entry__.build() where /root/reference exists)"}))
        return
    sys.path.insert(0, REF)
    sys.path.append(ROOT)            # only for sketchedit_b200.synth and oracle.golden; `models` resolves to _ref
    from argparse import Namespace

    import torch
    from models.editline2_model import EditLine2Model
    import models as ref_models
    assert os.path.realpath(ref_models.__file__).startswith(os.path.realpath(REF)), ref_models.__file__
    from oracle.golden import Golden
    from sketchedit_b200 import synth

    opt = Namespace(gpu_ids=[], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02,
                    continue_train=False, use_cam=True, pool_type="max", no_mask_cc=False, no_mask_coarse=False,
                    joint_train_inp=True)
    model = EditLine2Model(opt)
    model.netM.load_state_dict(synth.synth_state_dict("M"))
    model.netG.load_state_dict(synth.synth_state_dict("G"))
    model.eval()

    def fwd(image, sketch):
        data = {"image": image, "gt": image, "mask": sketch, "edgegt": sketch}
        with torch.no_grad():
            return model(data, mode="inference")

    base_img, base_sk = synth.synth_inputs(min(args.batch, 8), args.size, args.size, seed=0)
    reps = (args.batch + base_img.shape[0] - 1) // base_img.shape[0]
    img = base_img.repeat(reps, 1, 1, 1)[:args.batch].contiguous()
    sk = base_sk.repeat(reps, 1, 1, 1)[:args.batch].contiguous()

    ncpu = os.cpu_count() or 1
    threads = args.threads
    if threads <= 0:      # torch's CPU convolutions stop scaling well before 100+ threads at small batch: take the fastest
        best, best_t = None, float("inf")
        for t in sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu}):
            torch.set_num_threads(t)
            fwd(img[:1], sk[:1])
            t0 = time.perf_counter()
            fwd(img[:1], sk[:1])
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = t, dt
        threads = best
    torch.set_num_threads(threads)
    for _ in range(args.warmup):
        fwd(img, sk)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fwd(img, sk)
    dt = (time.perf_counter() - t0) / args.steps
    out = {"ok": True, "kind": "reference", "images_per_s": args.batch / dt, "s_per_step": dt, "threads": threads, "cores": ncpu,
           "batch": args.batch, "size": args.size}
    if args.face:
        g = Golden(os.path.join(ROOT, "tests", "golden", "face_602_256x256.npz"))
        fimg, fsk = g.inputs()
        comp, _ = fwd(fimg, fsk)
        t0 = time.perf_counter()
        for _ in range(3):
            comp, _ = fwd(fimg, fsk)
        out["face_b1_s"] = (time.perf_counter() - t0) / 3
        out["face_b1_max_abs_vs_golden"] = g.maxdiff("composed", comp)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
