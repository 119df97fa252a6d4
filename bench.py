"""Benchmark of the SketchEdit generator forward pass (BASELINE.json metric: images/sec, 256x256
CelebA-HQ-shaped inputs, synthetic seeded weights of the real architecture).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dtype bf16|fp32] [--batch B] [--size S]

One "step" = one forward of `model(data, mode='inference')` (netM + threshold + netG incl. contextual
attention + blend) over one batch. Default workload = BASELINE.json configs[2]: 256x256, batch 128 per GPU, bf16
tensor-core path (== the per-GPU shard of configs[4], 1024 images over 8 GPUs; weak scaling). `--dtype fp32
--batch 32` runs configs[1] (fp32 parity path); `--size 512 --batch 16` runs configs[3] (Places-size inputs,
contextual attention over L = 3969 patches).

Prints ONE JSON line (rank 0):
  value     whole-job throughput, inputs resident in HBM, NO instrumentation inside the timed region
  e2e       same metric through the reference-facing module API with pinned host tensors in and host tensors out
            (N > 1: including the NCCL all-gather of the outputs)
  roofline  from ONE separate instrumented pass (CUDA events around every launch, se_timing_enable): all tcgen05
            launches together, the dominant kernel class, and the per-class table with each class's own bound
  latency   batch-1 forward latency at 256x256 and 512x512 (N = 1, default workload only)
`--impl reference` times the UNMODIFIED reference (baseline/_ref, staged by __graft_entry__.build()) on the host cores
through baseline/ref_runner.py; if it was never staged, the CPU oracle port (kind "port").

`--dump-outputs DIR` writes what the last timed step returned (composed [N,3,H,W] and mask [N,1,H,W], float32) as
DIR/composed.npy and DIR/mask.npy, so that two builds can be compared output for output: inputs and weights are seeded, so
the same arguments give the same inputs on every run. On several GPUs N is the all-gathered global batch. When the outputs
exceed DUMP_BYTES, the same seeded sample of whole images is written for both. DIR/batch_index.txt lists, one per line, the
batch index of each dumped image; image i of a batch has the inputs of image i % 8 (make_inputs repeats 8 base images).
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNIT = "images/s"
DUMP_BYTES = 64 * 10 ** 6


def metric_name(size):
    return "images/sec %dx%d %s generator fwd" % (size, size, "CelebA-HQ" if size == 256 else "Places")


def workload_name(dtype, batch, n, size):
    return "%s %dx%d generator fwd (netM+netG+CAM), batch %d/GPU x %d GPU, %s, synthetic weights+inputs" % (
        "CelebA-HQ" if size == 256 else "Places", size, size, batch, n, dtype)


def make_inputs(batch, size):
    from sketchedit_b200 import synth
    base_img, base_sk = synth.synth_inputs(8, size, size, seed=0)
    reps = (batch + 7) // 8
    return base_img.repeat(reps, 1, 1, 1)[:batch].contiguous(), base_sk.repeat(reps, 1, 1, 1)[:batch].contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 25 ms during the timed regions (device-resident + e2e)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    PERIOD_MS = 25

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", str(self.PERIOD_MS)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference(size, n_img, steps, warm, face=False, threads=0):
    """The UNMODIFIED reference on the host cores (baseline/_ref through baseline/ref_runner.py, own process: its
    packages are called `models` / `util` like this repo's). Returns the runner's dict or None if it was never staged."""
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_runner.py"), "--size", str(size), "--batch", str(n_img), "--steps", str(steps),
           "--warmup", str(warm), "--threads", str(threads)] + (["--face"] if face else [])
    try:
        out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=900).stdout
        d = json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1])
        return d if d.get("ok") else None
    except Exception:
        return None


def cpu_port(size, n_img, steps, warm):
    """Fallback: the CPU oracle port of the reference path (oracle/), when baseline/_ref is absent."""
    from oracle import sketchedit_oracle as O
    from sketchedit_b200 import synth
    WM, WG = synth.synth_state_dict("M"), synth.synth_state_dict("G")
    ncpu = os.cpu_count() or 1
    img, sk = make_inputs(n_img, size)
    best, best_t = 8, float("inf")
    for t in sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu}):
        torch.set_num_threads(t)
        O.inference(WM, WG, img[:1], sk[:1])
        t0 = time.perf_counter()
        O.inference(WM, WG, img[:1], sk[:1])
        if time.perf_counter() - t0 < best_t:
            best, best_t = t, time.perf_counter() - t0
    torch.set_num_threads(best)
    for _ in range(warm):
        O.inference(WM, WG, img, sk)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.inference(WM, WG, img, sk)
    dt = (time.perf_counter() - t0) / steps
    return {"ok": True, "kind": "port", "images_per_s": n_img / dt, "s_per_step": dt, "threads": best, "cores": ncpu, "batch": n_img, "size": size}


def cpu_arm(size, n_img, steps, warm, face=False):
    d = cpu_reference(size, n_img, steps, warm, face=face)
    return d if d is not None else cpu_port(size, n_img, steps, warm)


def cpu_baseline_entry(d):
    what = ("the UNMODIFIED reference EditLine2Model (baseline/_ref), model(data, mode='inference')" if d["kind"] == "reference"
            else "torch CPU fp32 oracle port of the reference forward (baseline/_ref not staged)")
    e = {"value": d["images_per_s"], "unit": UNIT, "cores": d["threads"], "kind": d["kind"],
         "sample": "%s: batch %d of the workload at %dx%d, fp32, %d intra-op threads (fastest of a calibration over 8..%d host cores)" % (
             what, d["batch"], d["size"], d["size"], d["threads"], d["cores"])}
    if "face_b1_s" in d:
        e["config1_face602_b1"] = {"s_per_image": d["face_b1_s"], "images_per_s": 1.0 / d["face_b1_s"],
                                   "max_abs_vs_golden": d.get("face_b1_max_abs_vs_golden")}
    return e


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_img = 4 if args.size <= 256 else 1     # one step = a bounded slice of the workload batch
    d = cpu_arm(args.size, n_img, args.steps, args.warmup, face=(args.size == 256))
    line = {
        "impl": "reference", "metric": metric_name(args.size), "value": d["images_per_s"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": d["s_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": workload_name(args.dtype, args.batch, args.gpus, args.size), "step": "%d-image slice per step on CPU" % n_img},
        "cpu_baseline": cpu_baseline_entry(d),
        "e2e": {"value": d["images_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ roofline
def timing_report(lib):
    from sketchedit_b200 import _lib
    buf = ctypes.create_string_buffer(1 << 20)
    n = lib.se_timing_report(buf, len(buf))
    if n < 0:
        _lib.check(1)
    return json.loads(buf.value.decode())["classes"]


def roofline_from_classes(classes, steps, peaks, src, step_ms):
    """classes: se_timing_report rows over `steps` instrumented steps. Per class: bound = whichever of
    (algorithmic FLOPs / sustained bf16 peak, algorithmic bytes / HBM peak) takes longer; frac = that ideal time / measured."""
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    peak_bw = float(peaks["hbm_gbs"])
    rows, t_ideal_sum, t_sum = [], 0.0, 0.0
    for c in classes:
        ms = c["ms"] / steps
        if ms <= 0:
            continue
        fa, fe, by = c["flops_alg"] / steps, c["flops_exec"] / steps, c["bytes_alg"] / steps
        t_f, t_b = fa / (peak_tf * 1e12) * 1e3, by / (peak_bw * 1e9) * 1e3
        bound = "tensor" if (c["tensor"] and t_f >= t_b) else "hbm"
        ideal = t_f if bound == "tensor" else t_b
        t_ideal_sum += ideal
        t_sum += ms
        rows.append({"class": c["name"], "launches_per_step": c["launches"] / steps, "us_per_step": ms * 1e3, "bound": bound,
                     "tflops_alg": fa / ms / 1e9, "tflops_exec": fe / ms / 1e9, "gbs_alg": by / ms / 1e6, "frac": ideal / ms,
                     "tcgen05": bool(c["tensor"])})
    rows.sort(key=lambda r: -r["us_per_step"])
    tc = [r for r in rows if r["tcgen05"]]
    tc_ms = sum(r["us_per_step"] for r in tc) / 1e3
    tc_fa = sum(r["tflops_alg"] * r["us_per_step"] for r in tc) / 1e3      # TFLOP/s * ms = GFLOP... keep consistent below
    tc_fe = sum(r["tflops_exec"] * r["us_per_step"] for r in tc) / 1e3
    ach_alg = tc_fa / tc_ms if tc_ms else 0.0
    ach_exec = tc_fe / tc_ms if tc_ms else 0.0
    dom = tc[0] if tc else None
    roof = {
        "bound": "tensor", "kernel": "all tcgen05 launches (conv_c8_kernel classes: gated convs; cam_s / cam_pv or gemm_split: attention GEMMs)",
        "achieved": ach_alg, "achieved_executed": ach_exec, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_alg / peak_tf,
        "frac_executed": ach_exec / peak_tf,
        "flops_convention": "achieved = ALGORITHMIC 2*MAC of the reference ops the forward executes (SURVEY.md 8d; mode='inference' skips the dead netM "
                            "image decoder) / summed launch time; achieved_executed counts the MACs this implementation issues (sub-pixel deconvs: 4/9)",
        "peak_source": "%s bf16_tflops_sustained (kernels timed inside a long step)" % src,
        "kernel_share_of_step": tc_ms / step_ms, "instrumented_ms_per_step": t_sum,
        "per_layer_roofline_frac": t_ideal_sum / t_sum if t_sum else None,
        "per_layer_note": "sum over ALL launches of max(alg FLOPs / sustained bf16 peak, alg bytes / measured HBM GB/s) divided by the summed measured "
                          "launch time (north_star's 'per-layer tensor-core/HBM roofline')",
        "traffic": None,
        "dominant": dom and {k: dom[k] for k in ("class", "launches_per_step", "us_per_step", "tflops_alg", "frac")},
        "per_class": [[r["class"], round(r["launches_per_step"], 2), round(r["us_per_step"], 1), r["bound"],
                       round(r["tflops_alg"], 1) if r["bound"] == "tensor" else round(r["gbs_alg"], 1), round(r["frac"], 3)] for r in rows],
        "per_class_columns": ["class", "launches/step", "us/step", "bound", "TFLOP/s (tensor) or GB/s (hbm), algorithmic", "frac of its bound"],
    }
    return roof, rows


def load_traffic(workload_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture of this workload (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    e = d.get(workload_key)
    return (e["bytes_per_launch"], e["note"]) if e else (None, None)


def dump_outputs(out_dir, outputs):
    """outputs: {name: host tensor [N, C, H, W]} -> out_dir/<name>.npy (float32). Over DUMP_BYTES in all, every array keeps the
    same seeded sample of its N images; out_dir/batch_index.txt lists the batch index of each image kept."""
    import numpy as np
    n = next(iter(outputs.values())).shape[0]
    per_image = sum(t[0].numel() * 4 for t in outputs.values())
    keep = min(n, DUMP_BYTES // per_image)
    if keep == 0:
        raise SystemExit("--dump-outputs: one image's outputs (%d bytes) exceed the %d-byte limit" % (per_image, DUMP_BYTES))
    idx = np.arange(n) if keep == n else np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy()[idx].astype(np.float32))
    with open(os.path.join(out_dir, "batch_index.txt"), "w") as f:
        f.write("".join("%d\n" % i for i in idx))
    return idx


def write_class_table(path, rows, header):
    with open(path, "w") as f:
        f.write(header + "\n\n| us/step | launches/step | class | bound | achieved (algorithmic) | frac of bound |\n|---:|---:|---|---|---:|---:|\n")
        for r in rows:
            ach = "%.1f TFLOP/s (exec %.1f)" % (r["tflops_alg"], r["tflops_exec"]) if r["bound"] == "tensor" else "%.1f GB/s" % r["gbs_alg"]
            f.write("| %.1f | %.2f | `%s` | %s | %s | %.3f |\n" % (r["us_per_step"], r["launches_per_step"], r["class"], r["bound"], ach, r["frac"]))


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import torch.distributed as dist
    from argparse import Namespace

    import models
    from sketchedit_b200 import _lib, synth
    from sketchedit_b200.arch import cam_flops_per_image, conv_flops_per_image, dead_flops_per_image

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU for --impl b200 (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    B, H, W = args.batch, args.size, args.size
    prec = args.dtype

    opt = Namespace(gpu_ids=[local], isTrain=False, isSkip=True, netG="deepfillc2", init_type="xavier", init_variance=0.02,
                    use_cam=True, pool_type="max", no_mask_cc=False, no_mask_coarse=False, joint_train_inp=True,
                    model="editline2", precision=prec)
    model = models.create_model(opt)
    model.netM.load_state_dict(synth.synth_state_dict("M"))
    model.netG.load_state_dict(synth.synth_state_dict("G"))
    model.eval()
    eng = model.engine()
    lib = _lib.load()

    img_h, sk_h = make_inputs(B, args.size)          # each rank: its own contiguous shard (same synthetic content)
    img_h, sk_h = img_h.pin_memory(), sk_h.pin_memory()
    img_d, sk_d = img_h.cuda(non_blocking=True), sk_h.cuda(non_blocking=True)

    from sketchedit_b200 import parallel
    gather = parallel.OutputGather(B, H, W, torch.device("cuda", local)) if world > 1 else None

    def step_device():
        if gather is not None:      # heads write straight into this rank's slice of the gather buffer; the all-gather of
            slot = gather.next_slot()            # step i runs on NCCL's stream while step i+1 computes
            eng.inference_packed(img_d, sk_d, precision=prec, out=slot)
            gather.launch()
            return None
        return eng.inference(img_d, sk_d, precision=prec)[:2]

    def barrier():
        if gather is not None:
            gather.wait()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        last = step_device()        # held like in the timed loop: both output allocations are cached before it
    barrier()
    launches_per_step = eng.launches()

    # ---------------- timed region: device-resident inputs, no instrumentation
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step_device()
    if gather is not None:
        last = parallel.unpack_outputs(gather.wait())      # the last step's collective belongs to the region
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:     # before the passes below reuse the gather ring
        kept = dump_outputs(args.dump_outputs, {"composed": last[0].cpu(), "mask": last[1].cpu()})
        print("bench: wrote the last timed step's outputs (%d of %d images) to %s" % (len(kept), last[0].shape[0], args.dump_outputs),
              file=sys.stderr)
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * args.steps / (ms / 1e3)

    # ---------------- e2e: reference-facing module API, pinned host tensors in, host tensors out
    comp_h = torch.empty(B, 3, H, W).pin_memory()
    mask_h = torch.empty(B, 1, H, W).pin_memory()

    def step_e2e():
        with torch.no_grad():
            composed, mask = model({"image": img_h, "mask": sk_h}, mode="inference")
        comp_h.copy_(composed, non_blocking=True)
        mask_h.copy_(mask, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn):
        barrier()
        t0 = time.perf_counter()
        fn()
        barrier()
        t = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # (a) one blocking call per batch, as the reference's test.py loop does
    for _ in range(2):
        step_e2e()
    e2e_serial = world * B * args.steps / timed(lambda: [step_e2e() for _ in range(args.steps)])

    # (b) the package's pipelined loop over the same batches (models.EditLine2Model.inference_stream): every step copies its
    # own inputs host->device and its own outputs device->host on side streams. N = 1: the uint8 form (the codecs of the
    # reference's dataset / test.py run on the device: uint8 pixels in, uint8 BGR + mask out - what test.py drives). N > 1:
    # float tensors, and every step's outputs also go through the all-gather (gather=...) before they are copied out
    img_u8 = ((img_h.permute(0, 2, 3, 1) + 1) / 2 * 255).round().clamp(0, 255).to(torch.uint8).contiguous().pin_memory()
    sk_u8 = (sk_h[:, 0] * 255).to(torch.uint8).contiguous().pin_memory()

    def run_stream(n, u8):
        batch = {"image_u8": img_u8, "mask_u8": sk_u8} if u8 else {"image": img_h, "mask": sk_h}
        with torch.no_grad():
            for a, b in model.inference_stream((batch for _ in range(n)), gather=None if u8 else gather, uint8=u8):
                pass
        return a, b

    use_u8 = world == 1
    run_stream(6, use_u8)   # > depth + 2 batches: the pinned output ring is allocated (cudaHostAlloc is slow) before the timed loop
    e2e_value = world * B * args.steps / timed(lambda: run_stream(args.steps, use_u8))
    e2e_float = None
    if use_u8:
        run_stream(6, False)
        e2e_float = world * B * args.steps / timed(lambda: run_stream(args.steps, False))
    clocks = sampler.stop() if rank == 0 else None
    h2d = B * H * W * (4 if use_u8 else 16)
    d2h = B * H * W * (4 if use_u8 else 16)

    # ---------------- one instrumented pass for the roofline table (CUDA events around every launch)
    roof = rows = None
    if rank == 0:
        n_inst = 2
        lib.se_timing_enable(1)
        for _ in range(n_inst):
            eng.inference(img_d, sk_d, precision=prec)
        torch.cuda.synchronize()
        classes = timing_report(lib)
        lib.se_timing_enable(0)
        peaks, src = measured_peaks()
        roof, rows = roofline_from_classes(classes, n_inst, peaks, src, ms / args.steps)
        wkey = "%s_b%d_%d" % (prec, B, args.size)
        roof["traffic"], tnote = load_traffic(wkey)
        if tnote:
            roof["traffic_note"] = tnote
        if args.classes_out:
            write_class_table(args.classes_out, rows, "# per-kernel-class roofline, %s (one instrumented pass of %d steps, CUDA events per launch)" % (
                workload_name(prec, B, world, args.size), n_inst))

    # ---------------- batch-1 latency (config 1 shape) at 256x256 and 512x512
    latency = None
    if rank == 0 and world == 1 and not args.no_latency:
        latency = {}
        for s in (256, 512):
            im1, sk1 = make_inputs(1, s)
            im1, sk1 = im1.cuda(), sk1.cuda()
            for _ in range(5):
                eng.inference(im1, sk1, precision=prec)
            torch.cuda.synchronize()
            ts = []
            for _ in range(20):
                t0 = time.perf_counter()
                eng.inference(im1, sk1, precision=prec)
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            latency["b1_%dx%d_ms" % (s, s)] = {"median": statistics.median(ts), "min": min(ts)}
        latency["how"] = "wall clock around one blocking Engine.inference call + synchronize, device-resident input, 20 calls after 5 warm-ups"

    if rank == 0:
        cpu = cpu_arm(args.size, 4 if args.size <= 256 else 1, 2, 1, face=(args.size == 256)) if world == 1 else None
        alg = (conv_flops_per_image(H, W) + cam_flops_per_image(H, W)) / 1e9
        line = {
            "metric": metric_name(args.size), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": prec, "data": "synthetic",
            "config": {"workload": workload_name(prec, B, world, args.size), "global_batch": world * B, "H": H, "W": W,
                       "l2": "inputs + per-step activations (%.1f GB workspace) far exceed the 126 MB L2; no explicit flush" % (eng.workspace_bytes() / 1e9),
                       "parallelism": "dp%d (batch shards; one NCCL all-gather of the packed outputs per step, overlapped with the next step)" % world if world > 1 else "single GPU",
                       "algorithmic_gflop_per_image_reference": alg,
                       "algorithmic_gflop_per_image_executed_layers": alg - dead_flops_per_image(H, W) / 1e9,
                       "gflop_note": "mode='inference' never uses netM's image decoder (conv11-17, reference editline2_model.py:128-133): those "
                                     "%.2f GFLOP/img are not executed and not counted in roofline.achieved" % (dead_flops_per_image(H, W) / 1e9)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": ("models.create_model(opt).inference_stream(batches, uint8=True): pinned uint8 pixels in (dataset format before "
                            "ToTensor/Normalize) -> pinned uint8 BGR + mask out (test.py's output format), codecs on the device, per-step H2D/D2H "
                            "on side streams overlapping compute") if use_u8 else
                           ("models.create_model(opt).inference_stream(batches, gather=...): pinned float CPU tensors in -> pinned CPU outputs, "
                            "per-step H2D/D2H on side streams; outputs all-gathered over NCCL every step"),
                    "float_value": e2e_float,
                    "float_api": "same stream API with fp32 tensors (16 B per pixel each way)" if use_u8 else None,
                    "serial_value": e2e_serial,
                    "serial_api": "models.create_model(opt)(data, mode='inference') + .copy_ to pinned CPU, one blocking call per batch"},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roof,
        }
        if latency:
            line["latency"] = latency
        if cpu is not None:
            line["cpu_baseline"] = cpu_baseline_entry(cpu)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--dtype", default="bf16", choices=("bf16", "fp32"))
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default 128 bf16 / 32 fp32 at 256; 16 at 512)")
    ap.add_argument("--size", type=int, default=256, help="H = W of the synthetic inputs (256: CelebA-HQ configs, 512: Places config)")
    ap.add_argument("--classes-out", default=None, help="write the per-kernel-class roofline table (markdown) here")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the last timed step's outputs as DIR/<name>.npy (float32, a seeded sample of images beyond 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.batch is None:
        args.batch = 16 if args.size >= 512 else (128 if args.dtype == "bf16" else 32)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
