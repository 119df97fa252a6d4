"""Per-request latency and requests/s of DemoProcessor.process_image (the reference's demo.py:39-73 flow) with the three Pillow
resizes on the host (resize="host") and on the device (resize="device"), for a 637x477 request from 1 and from 16 client threads,
bf16. The two modes alternate within each thread count, `--repeats` times, so a drift of the shared host shows in both.

    python tools/demo_latency.py [--requests 400] [--repeats 2] [--max-wait-ms 2.0]

Prints one JSON line. The host side is what the modes change, so the line names the host CPU next to the GPU and its power limit.
"""
import argparse
import json
import os
import platform
import subprocess
import sys
import threading
import time
from argparse import Namespace

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import PIL  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

import models  # noqa: E402
from sketchedit_b200 import synth  # noqa: E402
from sketchedit_b200.serving import DemoProcessor  # noqa: E402

W, H = 637, 477


def host_cpu():
    name = platform.processor() or platform.machine()
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    name = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return {"model": name, "logical_cpus": os.cpu_count(), "usable_cpus": len(os.sched_getaffinity(0))}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(out[0]), sm_max_mhz=float(out[1]))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def make_model():
    opt = Namespace(gpu_ids=[0], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02, use_cam=True,
                    pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True, model="editline2", precision="bf16")
    model = models.create_model(opt)
    model.netM.load_state_dict(synth.synth_state_dict("M"))
    model.netG.load_state_dict(synth.synth_state_dict("G"))
    return model.eval()


def make_request(seed):
    rs = np.random.RandomState(seed)
    img = Image.fromarray(rs.randint(0, 256, (H, W, 3), dtype=np.uint8))
    m = np.zeros((H, W), np.uint8)
    m[100:380, 200 + seed % 50:204 + seed % 50] = 255
    m[240:244, 120:520] = 255
    return img, Image.fromarray(m)


def measure(proc, threads, requests):
    """`requests` process_image calls spread over `threads` client threads -> latencies (ms) and requests/s."""
    per = [requests // threads + (i < requests % threads) for i in range(threads)]
    reqs = [make_request(i) for i in range(threads)]
    lat = [[] for _ in range(threads)]
    start = threading.Barrier(threads + 1)

    def client(i):
        start.wait()
        for _ in range(per[i]):
            t0 = time.perf_counter()
            proc.process_image(*reqs[i])
            lat[i].append((time.perf_counter() - t0) * 1e3)

    ts = [threading.Thread(target=client, args=(i,)) for i in range(threads)]
    [t.start() for t in ts]
    start.wait()
    t0 = time.perf_counter()
    [t.join() for t in ts]
    wall = time.perf_counter() - t0
    all_lat = np.concatenate([np.array(v) for v in lat])
    return {"requests": int(all_lat.size), "requests_per_s": round(all_lat.size / wall, 1), "latency_ms_mean": round(float(all_lat.mean()), 3),
            "latency_ms_p50": round(float(np.percentile(all_lat, 50)), 3), "latency_ms_p90": round(float(np.percentile(all_lat, 90)), 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--requests", type=int, default=400, help="timed requests per (mode, thread count, repeat)")
    ap.add_argument("--warmup", type=int, default=32, help="untimed requests before each timed window")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--threads", default="1,16")
    ap.add_argument("--max-wait-ms", type=float, default=2.0, help="DemoProcessor batching window")
    ap.add_argument("--max-batch", type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("demo_latency.py measures the device path: it needs a CUDA device")
    torch.cuda.set_device(0)
    model = make_model()
    procs = {m: DemoProcessor(model, max_batch=args.max_batch, max_wait_ms=args.max_wait_ms, resize=m) for m in ("host", "device")}
    a, b = (np.array(procs[m].process_image(*make_request(0))) for m in ("host", "device"))
    runs = []
    for threads in (int(t) for t in args.threads.split(",")):
        for rep in range(args.repeats):
            for mode in ("host", "device"):
                measure(procs[mode], threads, args.warmup)
                runs.append(dict(mode=mode, threads=threads, repeat=rep, **measure(procs[mode], threads, args.requests)))
    for p in procs.values():
        p.close()
    print(json.dumps({"workload": "DemoProcessor.process_image %dx%d RGB + L mask, bf16" % (W, H), "max_batch": args.max_batch,
                      "max_wait_ms": args.max_wait_ms, "device_equals_host": bool(np.array_equal(a, b)), "gpu": gpu_info(),
                      "host_cpu": host_cpu(), "pillow": PIL.__version__, "torch": torch.__version__, "runs": runs}))


if __name__ == "__main__":
    main()
