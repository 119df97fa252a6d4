"""Throughput of the region inpaint (Engine.inpaint_u8: netG only) against the netM-predicted edit (Engine.inference_u8: netM +
netG) on the same seeded uint8 inputs, alternating the two entries in one process, for three workloads: bf16 256x256 batch 128,
bf16 512x512 batch 16 and fp32 (split-half tensor-core arithmetic) 256x256 batch 32.

    python tools/inpaint_throughput.py [--steps 50] [--warmup 5] [--rounds 3]

Every timed window runs `--steps` calls into the same device buffers (so they replay one captured CUDA graph) between two device
synchronisations. Inputs and outputs stay on the device: no PCIe copy is timed. Prints one JSON line with the GPU's name and power
limit read in the same run.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from sketchedit_b200 import synth  # noqa: E402
from sketchedit_b200.engine import Engine  # noqa: E402
from tools.demo_latency import gpu_info  # noqa: E402

WORKLOADS = [("bf16", 256, 128), ("bf16", 512, 16), ("fp32", 256, 32)]


def inputs(B, S, seed):
    """image RGB, sketch strokes (~3 % of pixels) and a region: each image's strokes dilated by a 31x31 box, i.e. a user circling them"""
    rs = np.random.RandomState(seed)
    img = torch.from_numpy(rs.randint(0, 256, (B, S, S, 3), dtype=np.uint8))
    sk = torch.zeros(B, S, S, dtype=torch.uint8)
    for b in range(B):
        for _ in range(4):
            y, x = rs.randint(S // 8, 7 * S // 8, size=2)
            sk[b, y:y + 2, max(0, x - S // 8):x + S // 8] = 255
            sk[b, max(0, y - S // 8):y + S // 8, x:x + 2] = 255
    rg = torch.nn.functional.max_pool2d(sk[:, None].float(), 31, stride=1, padding=15)[:, 0].to(torch.uint8)
    return img.cuda(), sk.cuda(), rg.cuda()


def window(fn, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50, help="calls per timed window")
    ap.add_argument("--warmup", type=int, default=5, help="untimed calls per entry and workload (>= 3: eager, capture, replay)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating (inference, inpaint) window pairs per workload")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("inpaint_throughput.py measures the device path: it needs a CUDA device")
    torch.cuda.set_device(0)
    eng = Engine.from_state_dicts(synth.synth_state_dict("M"), synth.synth_state_dict("G"))
    runs = []
    for prec, S, B in WORKLOADS:
        img, sk, rg = inputs(B, S, seed=S + B)
        bgr_a = torch.empty(B, S, S, 3, dtype=torch.uint8, device="cuda")
        bgr_b = torch.empty_like(bgr_a)
        mk = torch.empty(B, S, S, dtype=torch.uint8, device="cuda")
        entries = {"inference_u8": lambda: eng.inference_u8(img, sk, precision=prec, out=(bgr_a, mk)),
                   "inpaint_u8": lambda: eng.inpaint_u8(img, sk, rg, precision=prec, out=bgr_b)}
        for fn in entries.values():
            window(fn, args.warmup)
        rates = {k: [] for k in entries}
        for _ in range(args.rounds):
            for k, fn in entries.items():
                rates[k].append(B * args.steps / window(fn, args.steps))
        row = {"precision": prec, "size": S, "batch": B, "region_fraction": round(float((rg > 0).float().mean()), 4)}
        for k, v in rates.items():
            row[k + "_img_s"] = [round(r, 1) for r in v]
        row["inpaint_over_inference"] = round(float(np.mean(rates["inpaint_u8"]) / np.mean(rates["inference_u8"])), 3)
        runs.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    print(json.dumps({"workload": "inference_u8 vs inpaint_u8, seeded uint8 inputs on the device", "steps": args.steps,
                      "rounds": args.rounds, "gpu": gpu_info(), "torch": torch.__version__, "runs": runs}))


if __name__ == "__main__":
    main()
