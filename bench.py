#!/usr/bin/env python
"""Headline benchmark (driver contract in the task statement).

    python bench.py [--gpus N --steps K --warmup W]            the headline line (below)
    python bench.py --impl reference ...                        the reference arm: CPU oracle on all host cores
    python bench.py --workload clip|c4|c5 ...                   the other BASELINE.json configs as their own line

Headline workload at N GPUs: YOLOv9-c, 32 synthetic 640x640x3 uint8 BGR frames per GPU per step (BASELINE.json
configs[1], weak scaling: frames shard by batch, no data-path collective), whole path = stem(/255,BGR flip) -> 144 convs
-> DFL decode -> top-300 + suppression -> scale_boxes.  Weights: seeded synthetic (oracle.synthetic_weights).

  value     : frames/s with the uint8 frames already resident in HBM (rotating through > L2-size worth of inputs)
  e2e       : frames/s through the public API (YOLOv9.detect_pipelined) from PINNED HOST frames, H2D and the D2H read
              of the (B,300,6) result inside the timed region
  roofline  : conv_gemm_kernel (tcgen05) = algorithmic conv FLOPs per step / summed device time of its launches inside a
              plain forward (the kernels' own globaltimer stamps, cc_yolo_trace: no events between launches, PDL overlap as
              in the timed region), against MEASURED_PEAKS.json sustained bf16 peak; `frac_events` is the same with every
              launch bracketed by CUDA events (cc_yolo_profile: serialised, launch latency exposed)
  cpu_baseline / --impl reference : the torch-CPU oracle (the reference's tinygrad path cannot run here) on ALL host
              cores: `cpu_pool` starts cores/16 worker processes of 16 torch threads each (one oracle call does not scale
              past ~16 threads), releases them together and divides the units by the wall time of the slowest.  Both legs
              call the same function.
  clip      : the second hot loop (CLIP ViT-B/32 B=256, ViT-L/14 B=256, text tower) with its own value / e2e / roofline /
              cpu_baseline; `--workload clip` prints it as the line
  latency_b1: configs[0] — one 640x640 frame through `model(frame).numpy()` from pageable numpy, ms per call
  c4 / c5   : BASELINE configs[3] / [4] (multi-camera pipeline; YOLOv9-e + CLIP all-gather), emitted when N > 1 or on
              request

--dump-outputs DIR: after the timed steps, what the detector's and CLIP's timed paths returned in their last step, as
DIR/<name>.npy (float32; `.rank<r>` before `.npy` when N > 1): detections and e2e_detections (B,300,6), the detector head
of the last step's first two frames (2,84,anchors), and per CLIP tower <arch>_image_embeddings, <arch>_crop_embeddings and
<arch>_text_embeddings (256, embed_dim).  Weights and inputs are seeded, so two builds run with the same arguments can be
compared output for output.

oracle/ is imported here for three things only: the CPU legs, a small parity sample printed with the CPU leg, and — before
any timed region — the seeded synthetic weights and frames every arm runs on.  Every timed GPU region calls clearcam_b200
alone.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SIZE, RES, BATCH, HW = "c", 640, 32, 640
GFLOP_PER_FRAME = 102.14  # SURVEY.md §8(d), YOLOv9-c 640x640 (2*MAC over convs)
YOLO_WORKLOAD = (f"YOLOv9-c, {BATCH} uint8 {HW}x{HW}x3 BGR frames per GPU per step (BASELINE configs[1]), "
                 "stem->144 convs->DFL decode->top300+suppression->scale_boxes")
CLIP_WORKLOAD = "CLIP ViT-B/32 encode_image, 256 224x224x3 crops per GPU per step + encode_text (BASELINE configs[2])"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"tflops": p["bf16_tflops"], "tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm": p["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"tflops": 1590.0, "tflops_sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    def __init__(self, dev):
        self.dev, self.rows, self.proc = dev, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_weights(size=SIZE, hw=HW):
    from oracle import yolov9 as o
    fr = o.synthetic_frames(2, hw, hw, seed=0)
    x = fr.flip(-1).permute(0, 3, 1, 2).float() / 255
    return o.synthetic_weights(size, seed=0, calib=x)


# ------------------------------------------------------------------------------------------------ CPU legs
# One function serves `cpu_baseline` and `--impl reference`: same thread policy, same warm-up, same sample shape, so the two
# agree on the same box.  A single oracle call stops scaling at ~16 torch threads (128 threads were 10x SLOWER than 16 in
# round 1), so "all the host cores" means several worker processes of 16 threads each, working on different frames.
CPU_TASKS = {"yolo": {"units_per_call": 4, "unit": "frames/s"},          # 4 frames 640x640 through oracle.detect
             "clip": {"units_per_call": 8, "unit": "images/s"},          # 8 crops through oracle.clip.encode_image (ViT-B/32)
             "clip-text": {"units_per_call": 8, "unit": "queries/s"}}


def usable_cpus():
    """Host threads this process may actually use: the smaller of the visible CPUs, the affinity mask and the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    n = min(n, max(1, q // int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())))
        except Exception:
            pass
    return n


def cpu_policy():
    ncpu = usable_cpus()
    threads = min(16, ncpu)
    return max(1, min(8, ncpu // threads)), threads


def cpu_worker(args):
    """One worker of cpu_pool (spawned by it): load the shared weights, warm up, wait for the common start, run `steps`
    oracle calls, print its own start/end wall-clock times."""
    if args.pin:
        try:
            os.sched_setaffinity(0, {int(c) for c in args.pin.split(",")})
        except Exception:
            pass
    torch.set_num_threads(args.threads)
    task = args.cpu_worker
    P = torch.load(os.path.join(args.sync_dir, "weights.pt"))
    if task == "yolo":
        from oracle import yolov9 as o
        fr = o.synthetic_frames(4, HW, HW, seed=1 + args.worker_id)
        call = lambda: o.detect(SIZE, P, fr, RES)                            # noqa: E731
    else:
        from oracle import clip as oc
        cfg = oc.CONFIGS["ViT-B/32"]
        if task == "clip":
            x = oc.synthetic_images(8, cfg.image_size, seed=1 + args.worker_id)
            call = lambda: oc.encode_image(cfg, P, x)                         # noqa: E731
        else:
            g = torch.Generator().manual_seed(args.worker_id)
            ids = oc.pad_tokens([torch.randint(1000, 40000, (int(n),), generator=g).tolist() for n in torch.randint(3, 20, (8,), generator=g)])
            call = lambda: oc.encode_text_ids(cfg, P, ids)                    # noqa: E731
    with torch.no_grad():
        for _ in range(max(1, args.warmup)):
            call()
        open(os.path.join(args.sync_dir, f"ready.{args.worker_id}"), "w").close()
        go = os.path.join(args.sync_dir, "go")
        while not os.path.exists(go):
            time.sleep(0.002)
        t0 = time.time()
        for _ in range(args.steps):
            call()
        t1 = time.time()
    print(json.dumps({"t0": t0, "t1": t1, "calls": args.steps}), flush=True)


def _cpu_pool_run(task, d, nproc, threads, steps, warmup, pin):
    """Start `nproc` workers (optionally pinned to disjoint CPU sets), release them together, return (units/s, wall s)."""
    upc = CPU_TASKS[task]["units_per_call"]
    for f in os.listdir(d):
        if f.startswith("ready.") or f == "go":
            os.remove(os.path.join(d, f))
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads), CUDA_VISIBLE_DEVICES="")
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except Exception:
        cpus = list(range(os.cpu_count() or 1))
    procs = []
    for i in range(nproc):
        cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", task, "--threads", str(threads), "--steps", str(steps),
               "--warmup", str(warmup), "--sync-dir", d, "--worker-id", str(i)]
        if pin and len(cpus) >= nproc * threads:
            cmd += ["--pin", ",".join(str(c) for c in cpus[i * threads:(i + 1) * threads])]
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env))
    t_wait = time.time()
    while not all(os.path.exists(os.path.join(d, f"ready.{i}")) for i in range(nproc)):
        if any(p.poll() is not None for p in procs) or time.time() - t_wait > 900:
            errs = [p.communicate()[1][-2000:] for p in procs if p.poll() is not None]
            for p in procs:
                if p.poll() is None:
                    p.kill()
            raise RuntimeError("cpu_pool worker failed: " + " | ".join(errs))
        time.sleep(0.01)
    open(os.path.join(d, "go"), "w").close()
    outs = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in procs]
    wall = max(o["t1"] for o in outs) - min(o["t0"] for o in outs)
    return sum(o["calls"] for o in outs) * upc / wall, wall


def cpu_pool(task, P, steps, warmup=2):
    """units/s of the CPU oracle on the host cores this process may use.  Two layouts are timed with the same worker code and
    the FASTER one is reported (so the CPU leg is never handicapped by a bad layout): (a) usable/16 worker processes x 16 torch
    threads, pinned to disjoint CPU sets, `steps` calls each after `warmup` calls, released together (file barrier), units /
    (latest end - earliest start); (b) one worker of 16 threads alone (a single oracle call does not scale past ~16 threads)."""
    nproc, threads = cpu_policy()
    upc = CPU_TASKS[task]["units_per_call"]
    with tempfile.TemporaryDirectory(prefix="cc_cpu_") as d:
        torch.save(P, os.path.join(d, "weights.pt"))
        rate, wall = _cpu_pool_run(task, d, nproc, threads, steps, warmup, pin=True)
        layout = f"{nproc} pinned worker processes x {threads} torch threads"
        units = nproc * steps * upc
        if nproc > 1:
            r1, w1 = _cpu_pool_run(task, d, 1, threads, steps, warmup, pin=False)
            if r1 > rate:
                rate, wall, units = r1, w1, steps * upc
                layout = f"1 worker process x {threads} torch threads (faster than {nproc} workers x {threads} threads on this box)"
                nproc = 1
    return {"value": rate, "unit": CPU_TASKS[task]["unit"], "cores": nproc * threads, "kind": "port",
            "sample": f"{layout} of {usable_cpus()} usable host threads ({os.cpu_count()} visible), {units} units in {wall:.1f} s "
                      f"({upc} units per call, {warmup} warm-up calls)",
            "wall_s": wall, "steps": units // (nproc * upc), "units_per_step": nproc * upc}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, restated (oracle/): tinygrad DEV=CPU cannot
    run here.  A step = every worker runs one oracle call (4 frames / 8 crops)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    clip = args.workload == "clip"
    steps = args.steps
    warm = max(1, min(args.warmup, 3))
    if clip:
        from oracle import clip as oc
        P = oc.synthetic_weights(oc.CONFIGS["ViT-B/32"], seed=0)
        r = cpu_pool("clip", P, steps, warm)
        metric, workload = "images/s CLIP ViT-B/32 224px", CLIP_WORKLOAD
    else:
        r = cpu_pool("yolo", make_weights(), steps, warm)
        metric, workload = "frames/s YOLOv9-c 640px", YOLO_WORKLOAD
    line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": r["unit"], "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": warm, "ms_per_step": r["wall_s"] / r["steps"] * 1000, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "res": RES, "weights": "seeded synthetic",
                       "reference_arm": f"CPU oracle (torch fp32 restatement of the reference; tinygrad DEV=CPU cannot run here), "
                                        f"{r['units_per_step']} units per step"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": r["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def parity_sample(model, P):
    """Unconditioned deviation of the default (bf16-storage) CUDA path from the fp32 CPU oracle on 2 frames: every anchor's
    decoded box and class probabilities, no matching, no thresholds."""
    from oracle import yolov9 as o
    fr = o.synthetic_frames(2, HW, HW, seed=7)
    x = fr.flip(-1).permute(0, 3, 1, 2).float() / 255
    with torch.no_grad():
        want = o.forward_raw(SIZE, P, x)
    _, raw = model.detect_batch(fr, raw=True)
    got = raw.float().cpu()
    db = (got[:, :4] - want[:, :4]).abs().flatten()
    dp = (got[:, 4:] - want[:, 4:]).abs().flatten()
    q = lambda t, p: float(torch.quantile(t[:: max(1, t.numel() // 1000000)], p))    # noqa: E731
    return {"frames": 2, "vs": "fp32 CPU oracle, all anchors", "box_px": {"p50": q(db, 0.5), "p99": q(db, 0.99), "max": float(db.max())},
            "prob": {"p50": q(dp, 0.5), "p99": q(dp, 0.99), "max": float(dp.max())},
            "class_id_agreement": float((got[:, 4:].argmax(1) == want[:, 4:].argmax(1)).float().mean())}


# ------------------------------------------------------------------------------------------------ GPU sections
class Ctx:
    def __init__(self, args):
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
            # the seeded synthetic weights are generated on the CPU by every rank: share the host cores
            torch.set_num_threads(max(1, min(16, usable_cpus() // self.world)))
        else:
            torch.set_num_threads(min(16, usable_cpus()))
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        """barrier+sync, `steps` calls of fn(i) bracketed by CUDA events, barrier+sync, MAX over ranks -> total ms."""
        self.barrier()
        self.e0.record()
        for i in range(steps):
            fn(i)
        self.e1.record()
        self.barrier()
        t = torch.tensor([self.e0.elapsed_time(self.e1)], device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def dump(self, **arrays):
        """--dump-outputs: write each tensor as DIR/<name>.npy in float32."""
        d = self.args.dump_outputs
        if not d:
            return
        import numpy as np
        os.makedirs(d, exist_ok=True)
        sfx = f".rank{self.rank}" if self.world > 1 else ""
        for name, t in arrays.items():
            np.save(os.path.join(d, f"{name}{sfx}.npy"), t.detach().to("cpu", torch.float32).numpy())


def yolo_section(cx, with_cpu):
    from oracle import yolov9 as o
    from clearcam_b200.detection.yolov9 import YOLOv9
    args, world, rank = cx.args, cx.world, cx.rank
    B, W, K = args.batch, max(args.warmup, 3), args.steps
    P = make_weights()
    model = YOLOv9(SIZE, RES, weights=P)
    # > L2 (126 MB) worth of distinct device-resident input batches, rotated between steps
    nbuf = max(2, int(160e6 // (B * HW * HW * 3)) + 1)
    base = o.synthetic_frames(4, HW, HW, seed=100 + rank)
    g = torch.Generator(device="cuda").manual_seed(rank)
    dev_batches = []
    for i in range(nbuf):
        fb = base[torch.arange(B) % 4].cuda()
        noise = torch.randint(0, 8, fb.shape, device="cuda", dtype=torch.uint8, generator=g)
        dev_batches.append(((fb // 2) + noise + i).contiguous())
    host_batches = [b.cpu().pin_memory() for b in dev_batches[:2]]
    info = model.plan_info(B, HW, HW)

    # ---- device-resident throughput
    for i in range(W):
        model.detect_batch(dev_batches[i % nbuf])
    cx.barrier()
    sampler = ClockSampler(cx.local)
    if rank == 0:
        sampler.start()
    last = {}

    def step(i):
        last["detections"] = model.detect_batch(dev_batches[i % nbuf])
    ms_total = cx.timed(step, K)
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * K / (ms_total / 1000.0)

    # ---- end to end through the public API from pinned host memory
    for _ in model.detect_pipelined(host_batches[i % 2] for i in range(W)):
        pass
    n_out = [0]

    def e2e_all(_):
        for r in model.detect_pipelined(host_batches[i % 2] for i in range(K)):
            n_out[0] += r.shape[0]
            last["e2e_detections"] = r
    ms_e2e = cx.timed(e2e_all, 1)
    assert n_out[0] == B * K
    e2e = world * B * K / (ms_e2e / 1000.0)
    if args.dump_outputs:
        # these synthetic frames give few or no boxes above the 0.25 threshold (none in the last step at the defaults), so the
        # detections alone say little: add the head tensor they are selected from (boxes, class probabilities) for the last
        # step's input, frames 0 and 1
        _, raw = model.detect_batch(dev_batches[(K - 1) % nbuf], raw=True)
        last["head"] = raw[:2]
    cx.dump(**last)

    line = None
    if rank == 0:
        # ---- configs[0]: the reference's own call — one frame, pageable numpy in, numpy out (clearcam.py:580-583)
        f1 = base[0].numpy().copy()
        for _ in range(5):
            model(f1).numpy()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n1 = 30
        for _ in range(n1):
            model(f1).numpy()
        lat_ms = (time.perf_counter() - t0) / n1 * 1000

        # ---- roofline of the dominant kernel: live per-op CUDA-event timing + in-situ device timeline
        pk = peaks()
        prof = None
        for i in range(3):
            prof = model.profile(dev_batches[i % nbuf])
        by = {}
        for r in prof:
            d = by.setdefault(r["kind"], {"ms": 0.0, "flops": 0.0, "n": 0})
            d["ms"] += r["ms"]; d["flops"] += r["flops"]; d["n"] += 1
        gm = by.get("conv_gemm", {"ms": 1e-9, "flops": 0.0, "n": 0})
        # the memory-bound kernels: algorithmic bytes (inputs once + outputs once) / event-bracketed time, against the measured copy
        hbm = {}
        for r in prof:
            if r["kind"] != "conv_gemm" and r.get("bytes", 0) > 0:
                d = hbm.setdefault(r["kind"], {"ms": 0.0, "bytes": 0.0, "launches": 0})
                d["ms"] += r["ms"]; d["bytes"] += r["bytes"]; d["launches"] += 1
        for d in hbm.values():
            d["GB/s"] = d["bytes"] / (d["ms"] / 1000.0) / 1e9
            d["frac_of_hbm"] = d["GB/s"] / pk["hbm"]
            d["ms"] = round(d["ms"], 4); d["bytes"] = int(d["bytes"])
        achieved = gm["flops"] / (gm["ms"] / 1000.0) / 1e12
        total_prof_ms = sum(d["ms"] for d in by.values())
        try:
            tr = min((model.trace(dev_batches[i % nbuf]) for i in range(4)), key=lambda t: max(r["t_out"] for r in t))
            work_ms = sum(r["t_out"] - r["t_dep"] for r in tr if r["kind"] == "conv_gemm") / 1e6
            span_ms = max(r["t_out"] for r in tr) / 1e6
        except AttributeError:          # an older library under A/B comparison (tools/ab.py, CC_LIB) has no cc_yolo_trace
            work_ms = span_ms = float("nan")
        in_situ_tf = gm["flops"] / (work_ms / 1000.0) / 1e12
        # `achieved` / `frac`: algorithmic conv FLOPs of a step / the device time the conv kernels themselves take inside an
        # ordinary forward (production launch configuration: programmatic dependent launch, no host sync, no events between the
        # launches), read from globaltimer stamps the kernels write: per launch, last CTA exit - grid dependency released.  That
        # is what ncu's gpu__time_duration measures per launch, but warm and overlapped as in the timed region.
        # `frac_events` is the older figure: every launch bracketed by its own CUDA events, which serialises the stream and adds
        # the ~8 us launch latency to each of the 125 launches.
        roof = {"bound": "tensor", "kernel": "conv_gemm_kernel", "achieved": in_situ_tf, "peak": pk["tflops_sustained"],
                "unit": "TFLOP/s", "frac": in_situ_tf / pk["tflops_sustained"], "peak_src": pk["src"] + " (sustained bf16)",
                "how": "in-situ: globaltimer stamps written by the conv kernels (dependency released -> last CTA exit) during a plain forward, summed over the launches of a step",
                # DRAM bytes are not measurable without a profiler: see profiles/ for the ncu launch list of this command
                "traffic": None, "algorithmic_bytes": sum(r["bytes"] for r in prof if r["kind"] == "conv_gemm") / max(gm["n"], 1),
                "launches": gm["n"], "share_of_step": work_ms / (ms_total / K),
                "in_situ": {"conv_work_ms": work_ms, "first_conv_to_last_conv_ms": span_ms},
                "frac_events": achieved / pk["tflops_sustained"], "achieved_events": achieved,
                "share_of_step_events": gm["ms"] / total_prof_ms,
                "whole_step_tflops": B * GFLOP_PER_FRAME / 1000.0 / (ms_total / K / 1000.0),
                "whole_step_frac": B * GFLOP_PER_FRAME / 1000.0 / (ms_total / K / 1000.0) / pk["tflops_sustained"],
                "per_kind_ms_events": {k: round(v["ms"], 4) for k, v in by.items()},
                "memory_bound_kernels": {"peak": pk["hbm"], "unit": "GB/s", "peak_src": pk["src"] + " (copy)", "kernels": hbm}}
        cpu = None
        if with_cpu:                   # rank 0 at N=1 only: the other ranks must not sit in a barrier
            cpu = cpu_pool("yolo", P, steps=16, warmup=2)              # ~64 frames, ~10 s: the same order as the reference arm at the driver's K
            cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
            cpu["parity_sample"] = parity_sample(model, P)
        line = {"metric": "frames/s YOLOv9-c 640px", "value": value, "unit": "frames/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": YOLO_WORKLOAD if B == BATCH else YOLO_WORKLOAD.replace(f"{BATCH} uint8", f"{B} uint8"),
                           "global_batch": world * B, "res": RES, "weights": "seeded synthetic",
                           "l2": f"{nbuf} rotating input batches ({nbuf * B * HW * HW * 3 / 1e6:.0f} MB) + {info['act_bytes'] / 1e9:.1f} GB activations per step (> 126 MB L2)",
                           "parallelism": f"dp{world} (frames sharded by batch, no collective)"},
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * HW * HW * 3, "d2h_bytes_per_step": B * 300 * 6 * 4},
                "gpu_launches": info["launches"] * K,
                "latency_b1": {"ms": lat_ms, "frames_per_s": 1000.0 / lat_ms, "launches": model.plan_info(1, HW, HW)["launches"],
                               "how": "configs[0]: model(frame).numpy() on one pageable numpy 640x640x3 frame, wall clock over 30 calls"},
                "roofline": roof, "cpu_baseline": cpu}
    del model
    torch.cuda.empty_cache()
    return line


def clip_section(cx, with_cpu, archs=(("ViT-B/32", 256), ("ViT-L/14", 256))):
    """CLIP image + text towers: device-resident images/s, end to end from pinned host uint8 frames through
    ObjectFinder.embed_crops (H2D of the frames, device crop + bicubic + normalise, encoder, D2H of the embeddings), GEMM
    roofline from per-op events, text queries/s; all ranks, in-place all-gather of the embeddings when N > 1."""
    from oracle import clip as oc
    from oracle import yolov9 as oy
    from clearcam_b200.models.objects import ObjectFinder
    world, rank, K = cx.world, cx.rank, cx.args.steps
    pk = peaks()
    res = {}
    for arch, cb in archs:
        cfg = oc.CONFIGS[arch]
        P = oc.synthetic_weights(cfg, seed=0)
        fin = ObjectFinder()
        fin.init_clip(weights=P, arch=arch)
        cm = fin.model
        xs = [oc.synthetic_images(8, cfg.image_size, seed=10 + i)[torch.arange(cb) % 8].cuda() for i in range(3)]
        for i in range(3):
            cm.precompute_embedding(xs[i % 3], gather=world > 1)
        tag = arch.replace("ViT-", "vit_").replace("/", "").lower()          # ViT-B/32 -> vit_b32
        last = {}

        def image_step(i):
            last[f"{tag}_image_embeddings"] = cm.precompute_embedding(xs[i % 3], gather=world > 1).tensor
        ms = cx.timed(image_step, K)
        ips = world * cb * K / (ms / 1000.0)
        r = {"batch_per_gpu": cb, "value": ips, "unit": "images/s", "ms_per_step": ms / K,
             "tflops": ips * oc.flops_image(cfg) / 1e12, "gflop_per_image": oc.flops_image(cfg) / 1e9, "all_gather": world > 1}
        # e2e: 16 pinned host 720p frames, 16 object rectangles each (= cb crops) -> embeddings on the host
        nfr = 16
        per = cb // nfr
        hf = oy.synthetic_frames(2, 720, 1280, seed=3)[torch.arange(nfr) % 2].contiguous().pin_memory()
        gr = torch.Generator().manual_seed(5)
        rects = []
        for f in range(nfr):
            for _ in range(per):
                w, h = int(torch.randint(100, 400, (1,), generator=gr)), int(torch.randint(100, 400, (1,), generator=gr))
                x1, y1 = int(torch.randint(0, 1280 - w, (1,), generator=gr)), int(torch.randint(0, 720 - h, (1,), generator=gr))
                rects.append((f, x1, y1, x1 + w, y1 + h))
        hout = torch.empty(cb, cm.embed_dim, dtype=torch.float32, pin_memory=True)

        def e2e_step(_):
            dev = hf.to("cuda", non_blocking=True)
            hout.copy_(fin.embed_crops(dev, rects).tensor, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for _ in range(2):
            e2e_step(0)
        ms = cx.timed(e2e_step, K)
        last[f"{tag}_crop_embeddings"] = hout
        r["e2e"] = {"value": world * cb * K / (ms / 1000.0), "unit": "images/s", "h2d_bytes_per_step": hf.numel(),
                    "d2h_bytes_per_step": hout.numel() * 4,
                    "how": f"{nfr} pinned 720p uint8 frames + {cb} rectangles -> ObjectFinder.embed_crops -> pinned host embeddings, synchronous per step"}
        # text tower
        qb = 256
        g = torch.Generator().manual_seed(1)
        ids = oc.pad_tokens([torch.randint(1000, 40000, (int(n),), generator=g).tolist() for n in torch.randint(3, 20, (qb,), generator=g)]).int().cuda()
        for _ in range(2):
            cm.encode_token_ids(ids)

        def text_step(i):
            last[f"{tag}_text_embeddings"] = cm.encode_token_ids(ids).tensor
        ms = cx.timed(text_step, K)
        cx.dump(**last)
        r["text"] = {"batch_per_gpu": qb, "queries_per_s": world * qb * K / (ms / 1000.0),
                     "tflops": world * qb * K / (ms / 1000.0) * oc.flops_text(cfg) / 1e12}
        if rank == 0:
            cm._encode_text("a person walking a dog", realize=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                cm._encode_text("a person walking a dog", realize=True)      # the reference's speed probe, test/test_clip_speed.py:8-15
            r["text"]["single_query_ms"] = (time.perf_counter() - t0) / 20 * 1000
            ops, _tot = None, None
            for _ in range(2):
                ops, _tot = cm.profile(x=xs[0])
            r["launches_per_step"] = len(ops) + sum(1 for o_ in ops if o_["name"] == "attention")     # attention = V^T pre-pass + main kernel
            gemm = [o_ for o_ in ops if o_["name"] in ("qkv", "out_proj", "mlp_fc", "mlp_proj", "patch_embed", "proj")]
            attn = [o_ for o_ in ops if o_["name"] == "attention"]
            other = [o_ for o_ in ops if o_ not in gemm and o_ not in attn]
            gms, gfl = sum(o_["ms"] for o_ in gemm), sum(o_["flops"] for o_ in gemm)
            ams, afl = sum(o_["ms"] for o_ in attn), sum(o_["flops"] for o_ in attn)
            r["roofline"] = {"bound": "tensor", "kernel": "conv_gemm_kernel (QKV / out-proj / MLP GEMMs)", "achieved": gfl / gms / 1e9,
                             "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": gfl / gms / 1e9 / pk["tflops_sustained"],
                             "peak_src": pk["src"] + " (sustained bf16)", "traffic": None, "launches": len(gemm),
                             "share_of_step": gms / sum(o_["ms"] for o_ in ops),
                             "attention": {"ms": ams, "tflops": afl / max(ams, 1e-9) / 1e9, "share_of_step": ams / sum(o_["ms"] for o_ in ops)},
                             "other_kernels_ms": sum(o_["ms"] for o_ in other)}
            if with_cpu and arch == "ViT-B/32":
                c = cpu_pool("clip", P, steps=16, warmup=2)
                r["cpu_baseline"] = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
                c = cpu_pool("clip-text", P, steps=16, warmup=2)
                r["text"]["cpu_baseline"] = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
        res[arch] = r
        del cm, fin, xs, P
        torch.cuda.empty_cache()
    return res


def c4_section(cx):
    """BASELINE configs[3]: 8 synthetic 1080p camera feeds -> pinned frame mailboxes -> CameraBatch (letterbox to 384x640,
    YOLOv9-c, trackers) -> save_object rectangles of the detections -> device crop + CLIP ViT-B/32 embed -> all-gather of the
    embeddings.  The 8 cameras are sharded over the ranks (strong scaling: 8 frames per step in total)."""
    from oracle import clip as oc
    from oracle import yolov9 as o
    from clearcam_b200.cameras import CameraBatch
    from clearcam_b200.detection.yolov9 import YOLOv9
    from clearcam_b200.ingest import FrameMailbox
    from clearcam_b200.models.objects import ObjectFinder
    world, rank = cx.world, cx.rank
    NCAM, H, W = 8, 1080, 1920
    mine = [c for c in range(NCAM) if c % world == rank]
    model = YOLOv9(SIZE, RES, weights=make_weights())
    fin = ObjectFinder()
    fin.init_clip(weights=oc.synthetic_weights(oc.CONFIGS["ViT-B/32"], seed=0), arch="ViT-B/32")
    cb = CameraBatch(model)
    pool = o.synthetic_frames(3, H, W, seed=40 + rank)
    feeds = [[pool[(c + t) % 3].numpy().tobytes() for t in range(3)] for c in mine]
    boxes = {c: FrameMailbox(H, W) for c in mine}
    MAXC = 8                                     # at most 8 object crops per frame (bounds the synthetic detector's output)
    emb_local = torch.zeros(max(1, len(mine)) * MAXC, fin.model.embed_dim, device="cuda")
    emb_all = torch.zeros(world * emb_local.shape[0], fin.model.embed_dim, device="cuda") if world > 1 else None
    counts = {"frames": 0, "crops": 0}

    def step(t):
        for j, c in enumerate(mine):
            boxes[c].fill(io.BytesIO(feeds[j][t % 3]))                      # the ingest thread's job: bytes -> pinned slot
        res = cb.step_mailboxes(boxes)
        emb_local.zero_()
        row = 0
        for c, r in res.items():
            rects = []
            for d in r.rows[r.rows[:, 4] > 0][:MAXC]:
                q = ObjectFinder.crop_rect(d[:4], W, H)
                if q is not None:
                    rects.append(q)
            if rects:
                e = fin.embed_crops(cb.device_frame(c), rects).tensor     # the device copy the detector just read
                emb_local[row:row + len(rects)] = e
                row += len(rects)
            counts["frames"] += 1
        counts["crops"] += row
        if world > 1:
            cx.dist.all_gather_into_tensor(emb_all, emb_local)
    for t in range(3):
        step(t)
    counts["frames"] = counts["crops"] = 0
    K = cx.args.steps
    ms = cx.timed(step, K)
    tot = torch.tensor([counts["frames"], counts["crops"]], device="cuda", dtype=torch.float64)
    if world > 1:
        cx.dist.all_reduce(tot)
    out = {"workload": "8 x 1080p uint8 feeds -> mailboxes -> CameraBatch(YOLOv9-c @384x640 + OC-SORT) -> crop_rect -> embed_crops(ViT-B/32) -> all-gather",
           "scaling": "strong (8 cameras over the ranks)", "steps": K, "ms_per_step": ms / K,
           "frames_per_s": float(tot[0]) / (ms / 1000.0), "crops_per_s": float(tot[1]) / (ms / 1000.0),
           "h2d_bytes_per_step": NCAM * H * W * 3, "e2e": True,
           "note": "every step includes the host copy of each new frame into its pinned mailbox slot, H2D, the detector, the trackers (host C++), the crops' embeddings and the gather"}
    del model, fin, cb
    torch.cuda.empty_cache()
    return out


def c5_section(cx):
    """BASELINE configs[4]: YOLOv9-e, 16 frames 640x640 per GPU per step (128 over 8 GPUs) + CLIP ViT-B/32 embeddings of 2
    object crops per frame + NCCL all-gather of the embeddings (weak scaling)."""
    from oracle import clip as oc
    from oracle import yolov9 as o
    from clearcam_b200.detection.yolov9 import YOLOv9
    from clearcam_b200.models.objects import ObjectFinder
    world, rank = cx.world, cx.rank
    B = 16
    model = YOLOv9("e", RES, weights=make_weights("e"))
    fin = ObjectFinder()
    fin.init_clip(weights=oc.synthetic_weights(oc.CONFIGS["ViT-B/32"], seed=0), arch="ViT-B/32")
    base = o.synthetic_frames(4, HW, HW, seed=60 + rank)
    batches = [(base[torch.arange(B) % 4] // 2 + i).contiguous().cuda() for i in range(12)]      # 236 MB > L2
    rects = [(f, 40 + 10 * f, 60, 40 + 10 * f + 300, 60 + 360) for f in range(B)] + [(f, 200, 100 + 5 * f, 520, 420 + 5 * f) for f in range(B)]
    full = torch.empty(world * 2 * B, fin.model.embed_dim, device="cuda")

    def step(i):
        fb = batches[i % len(batches)]
        model.detect_batch(fb)
        x = fin.preprocess_device(fb, rects)
        fin.model.embed_into(x, full, rank * 2 * B)
        if world > 1:
            cx.dist.all_gather_into_tensor(full, full[rank * 2 * B:(rank + 1) * 2 * B])
    for i in range(3):
        step(i)
    K = cx.args.steps
    ms = cx.timed(step, K)
    fps = world * B * K / (ms / 1000.0)
    out = {"workload": f"YOLOv9-e, {B} uint8 640x640 frames per GPU per step ({world * B} in total) + ViT-B/32 embeddings of {2 * B} crops per GPU + all-gather",
           "scaling": "weak", "steps": K, "ms_per_step": ms / K, "frames_per_s": fps, "crops_per_s": 2 * fps,
           "tflops_detector": fps * 188.95 / 1000.0, "detector_frac_of_sustained": fps * 188.95 / 1000.0 / world / peaks()["tflops_sustained"]}
    del model, fin
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--workload", default="yolo", choices=["yolo", "clip", "c4", "c5"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-clip", action="store_true", help="headline line without the clip object")
    ap.add_argument("--extras", action="store_true", help="add the c4 and c5 objects to the headline line (default when N > 1)")
    ap.add_argument("--cpu-worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--threads", type=int, default=16, help=argparse.SUPPRESS)
    ap.add_argument("--sync-dir", default="", help=argparse.SUPPRESS)
    ap.add_argument("--worker-id", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--pin", default="", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs of the detector and CLIP paths as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("c4", "c5")):
        ap.error("--dump-outputs covers the detector and CLIP paths: workloads yolo and clip, not --impl reference")
    if args.cpu_worker:
        return cpu_worker(args)
    if args.impl == "reference":
        return run_reference(args)

    cx = Ctx(args)
    with_cpu = (not args.no_cpu) and cx.world == 1
    line = None
    if args.workload == "yolo":
        line = yolo_section(cx, with_cpu)
        extra = {}
        if not args.no_clip:
            try:
                extra["clip"] = clip_section(cx, with_cpu)
            except Exception as ex:                        # the detector line must still be printed
                extra["clip"] = {"error": repr(ex)}
        if args.extras or cx.world > 1:
            for name, fn in (("c4", c4_section), ("c5", c5_section)):
                try:
                    extra[name] = fn(cx)
                except Exception as ex:
                    extra[name] = {"error": repr(ex)}
        if line is not None:
            line.update(extra)
    elif args.workload == "clip":
        r = clip_section(cx, with_cpu)
        if cx.rank == 0:
            b = r["ViT-B/32"]
            line = {"metric": "images/s CLIP ViT-B/32 224px", "value": b["value"], "unit": "images/s", "n_gpus": cx.world,
                    "steps": args.steps, "warmup": 3, "ms_per_step": b["ms_per_step"], "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                    "config": {"workload": CLIP_WORKLOAD, "global_batch": cx.world * 256, "weights": "seeded synthetic",
                               "l2": "3 rotating input batches of 154 MB (> 126 MB L2)",
                               "parallelism": f"dp{cx.world} (crops sharded by batch; in-place all-gather of the embeddings when N > 1)"},
                    "e2e": b["e2e"], "roofline": b.get("roofline"), "cpu_baseline": b.get("cpu_baseline"), "text": b["text"],
                    "gpu_launches": b.get("launches_per_step", 0) * args.steps, "ViT-L/14": r["ViT-L/14"]}
    else:
        r = (c4_section if args.workload == "c4" else c5_section)(cx)
        if cx.rank == 0:
            line = {"metric": "frames/s " + ("8x1080p cameras detect+embed" if args.workload == "c4" else "YOLOv9-e 640px + CLIP all-gather"),
                    "value": r["frames_per_s"], "unit": "frames/s", "n_gpus": cx.world, "steps": r["steps"], "warmup": 3,
                    "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": r["scaling"].split()[0], "vs_baseline": None,
                    "dtype": "bf16", "data": "synthetic", "config": {"workload": r["workload"]}, args.workload: r}
    if cx.rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    if cx.dist is not None:
        cx.dist.barrier()
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
