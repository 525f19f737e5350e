#!/usr/bin/env python
"""Benchmark of the hot path: frames/sec end-to-end (rtpose VGG19 net + fused pafprocess) at 368x368.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...  (the reference algorithm on the host CPU cores)

One "step" = one pass of the hot path over one batch of 32 synthetic frames per GPU (BASELINE.json configs[2] /
configs[3]: batch 32 per B200, bf16, fused post-processing).  Weights: seeded He-normal (SURVEY.md 8c), inputs:
seeded uniform [-0.5, 0.5).  Prints ONE JSON line on rank 0.
"""
import argparse
import datetime
import importlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec end-to-end (net+pafprocess) @368x368"
UNIT = "frames/s"
BATCH, H, W = 32, 368, 368
FLOPS_PER_FRAME = 271868013568.0        # SURVEY.md 8(d): convolution FLOPs per 368x368 frame


def peaks(clocks):
    """Roofline denominators.  The burst figure applies when the kernel ran at the maximum SM clock with no power cap
    during the timed region (each launch is timed in isolation by an event pair and the region is short); the sustained
    figure applies when the clock sampler saw sw_power_cap or a median clock well below the maximum."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    capped = (clocks is None or "sw_power_cap" in (clocks.get("reasons") or []) or not clocks.get("sm_mhz")
              or clocks["sm_mhz"] < 0.97 * clocks.get("sm_max_mhz", 1965.0))
    if os.path.exists(p):
        d = json.load(open(p))
        tf = d.get("bf16_tflops_sustained", 1400.0) if capped else d.get("bf16_tflops", 1590.0)
        return tf, d.get("hbm_gbs", 6650.0), "of measured (MEASURED_PEAKS.json, %s)" % ("bf16_tflops_sustained: power cap / reduced clock seen"
                                                                                     if capped else "bf16_tflops burst: max SM clock, no power cap seen")
    return (1400.0 if capped else 1590.0), 6650.0, "of fallback (B200_PROFILING.md, %s)" % ("sustained" if capped else "burst")


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  Two sources, because the timed region of the default
    run is only ~0.2 s: an NVML thread (nvidia_ml_py) that samples every 10 ms between mark_start() and stop(), and an
    `nvidia-smi -lms 100` process started ahead of the warm-up whose time-stamped rows are filtered to the same window (the
    fallback when NVML is not importable; if no row falls inside the window the nearest one is used and named)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index, uuid=None):
        self.t0 = self.t1 = None
        self.nv_rows, self.nv_stop, self.nv_thread, self.nv_handle, self.nv = [], threading.Event(), None, None, None
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        # nvidia-smi / NVML count physical GPUs: the CUDA index only matches when CUDA_VISIBLE_DEVICES does not remap it
        remapped = bool(os.environ.get("CUDA_VISIBLE_DEVICES"))
        sel = str(uuid) if (uuid and remapped) else str(gpu_index)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", sel, "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.nv_handle = None
            if uuid and remapped:
                for u in (str(uuid), str(uuid).encode()):
                    try:
                        self.nv_handle = pynvml.nvmlDeviceGetHandleByUUID(u)
                        break
                    except Exception:
                        pass
            if self.nv_handle is None:
                self.nv_handle = pynvml.nvmlDeviceGetHandleByIndex(int(gpu_index))
            self.nv_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.nv_handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = self.nv_handle = None

    def _nv_loop(self):
        nv, h = self.nv, self.nv_handle
        while not self.nv_stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.nv_rows.append((sm, pw, rs))
            except Exception:
                break
            self.nv_stop.wait(0.01)

    def mark_start(self):
        self.t0 = datetime.datetime.now()
        if self.nv_handle is not None:
            self.nv_thread = threading.Thread(target=self._nv_loop, daemon=True)
            self.nv_thread.start()

    def stop(self):
        self.t1 = datetime.datetime.now()
        self.nv_stop.set()
        if self.nv_thread is not None:
            self.nv_thread.join(timeout=2)
        smi = self._stop_smi()
        if self.nv_rows:
            sm = [r[0] for r in self.nv_rows]
            reasons = sorted({name for r in self.nv_rows for bit, name in self.BITS if r[2] & bit})
            return {"sm_mhz": statistics.median(sm), "sm_max_mhz": self.nv_max, "power_w_max": round(max(r[1] for r in self.nv_rows), 2),
                    "samples": len(self.nv_rows), "reasons": reasons, "source": "nvml, every 10 ms inside the timed region"}
        return smi

    def _stop_smi(self):
        if self.p is None:
            return None
        time.sleep(0.12)                      # let the row that covers the end of the window be written
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = []
        for l in open(self.f.name).read().strip().splitlines():
            r = [c.strip() for c in l.split(",")]
            if len(r) < 9:
                continue
            try:
                rows.append((datetime.datetime.strptime(r[0], "%Y/%m/%d %H:%M:%S.%f"), r))
            except Exception:
                continue
        os.unlink(self.f.name)
        if not rows:
            return None
        t0 = self.t0 or rows[0][0]
        inside = [r for ts, r in rows if t0 <= ts <= self.t1]
        source = "nvidia-smi -lms 100, rows inside the timed region"
        if not inside:
            ts, r = min(rows, key=lambda x: abs((x[0] - t0).total_seconds()))
            inside = [r]
            source = "nvidia-smi: nearest row, %+.0f ms from the start of the timed region" % ((ts - t0).total_seconds() * 1e3)
        sm = [float(r[1]) for r in inside if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower() == "active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(inside[0][2]),
                "power_w_max": max(float(r[3]) for r in inside), "samples": len(inside), "reasons": sorted(reasons),
                "source": source}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, per_frame):
    """What the last timed step returns to a caller (PoseEngine.fetch_arrays): humans.npy, every person row
    [k, 73] (score, 18 x (x, y, peak score, peak id | -1)) of every frame in frame order, and humans_per_frame.npy.
    Above DUMP_BYTES the rows are a fixed seeded sample, and humans_index.npy names the rows kept."""
    os.makedirs(out_dir, exist_ok=True)
    counts = np.array([len(r) for r in per_frame], np.float64)
    rows = np.concatenate(per_frame).astype(np.float32)
    cap = (DUMP_BYTES - counts.nbytes) // (rows.shape[1] * rows.itemsize)
    if len(rows) > cap:
        keep = np.sort(np.random.RandomState(0).choice(len(rows), cap, replace=False))
        rows = rows[keep]
        np.save(os.path.join(out_dir, "humans_index.npy"), keep.astype(np.float64))
    np.save(os.path.join(out_dir, "humans.npy"), rows)
    np.save(os.path.join(out_dir, "humans_per_frame.npy"), counts)


def synthetic_weights():
    import _b200_alias
    return importlib.import_module(_b200_alias.PKG + ".synthetic").he_state_arrays(1234)


def run_ours(args):
    import torch
    import _b200_alias
    _b200_alias.load_package()
    engine = importlib.import_module(_b200_alias.PKG + ".engine")
    nat = importlib.import_module(_b200_alias.PKG + "._native")
    dist_mod = importlib.import_module(_b200_alias.PKG + ".distributed")
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL's version banner goes there)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        arrays = dist_mod.broadcast_state_arrays(synthetic_weights() if rank == 0 else None, device=dev)
    else:
        arrays = synthetic_weights()
    eng = engine.PoseEngine(arrays, local, mode=args.mode, batch_cap=BATCH, peak_cap=1024, human_cap=512)

    # Frames are uint8 HWC BGR (what cv2.imread / crop_with_factor hand to get_outputs); rtpose_preprocess is fused
    # into the first convolution.  10 rotating device batches (10 x 13 MB > 126 MB L2) + 2 pinned host batches.
    g = torch.Generator().manual_seed(1234 + rank)
    # --raw N: the frames are N x N "camera" frames and crop_with_factor (resize to 368 x 368) runs on the device too
    SH = SW = args.raw if args.raw else H          # (multi-scale: the raw frames are 368 x 368 unless --raw says otherwise)
    host = [torch.randint(0, 256, (BATCH, SH, SW, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    # enough rotating device batches that one full rotation exceeds the 126 MB L2 (10 at batch 32)
    n_rot = max(10, -(-130_000_000 // (BATCH * SH * SW * 3)))
    devin = [torch.randint(0, 256, (BATCH, SH, SW, 3), generator=g, dtype=torch.uint8).to(dev) for i in range(n_rot)]
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=dev)      # a real stream (not the legacy default): the forward pass replays as a CUDA graph
    torch.cuda.set_stream(stream)
    sptr = stream.cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    scales = [float(v) for v in args.scales.split(",")] if args.scales else None
    if scales:
        def infer_u8(ptr, on_device, n, h_, w_, thresh, stream):
            return eng.infer_raw_multiscale_async_u8(ptr, on_device, n, SH, SW, scales, H, 8, thresh, args.flip, stream)
    elif args.raw:
        def infer_u8(ptr, on_device, n, h_, w_, thresh, stream):
            return eng.infer_raw_async_u8(ptr, on_device, n, SH, SW, H, 8, thresh, args.flip, stream)
    else:
        infer_u8 = eng.infer_flip_async_u8 if args.flip else eng.infer_async_u8

    def step_device(i):
        infer_u8(devin[i % n_rot].data_ptr(), True, BATCH, H, W, 0.1, sptr)

    d2h_bytes = []

    def submit_e2e(i):
        return infer_u8(host[i % 2].data_ptr(), False, BATCH, H, W, 0.1, sptr)

    def fetch_e2e(ticket):
        eng.post.select(ticket)
        nh = 0
        for k in range(BATCH):
            nh += len(eng.post.humans(k))
        # what actually crosses PCIe per step: counts/status/n_humans + the person rows that exist (the assembly kernel
        # writes them straight into the pinned host slot)
        d2h_bytes.append(4 * BATCH * (1 + 1 + 18) + nh * 73 * 4)
        return nh

    sampler = None
    if rank == 0:       # (started ahead of the warm-up: nvidia-smi needs ~0.3 s to come up; only rows inside the timed region count)
        try:
            gpu_uuid = str(torch.cuda.get_device_properties(local).uuid)
            if not gpu_uuid.startswith("GPU-"):
                gpu_uuid = "GPU-" + gpu_uuid
        except Exception:
            gpu_uuid = None
        try:
            sampler = ClockSampler(local, gpu_uuid)
        except Exception:
            sampler = None
    for i in range(args.warmup):
        step_device(i)
    torch.cuda.synchronize()
    eng.post.status_accum(reset=True)     # from here on: OR of the status words of EVERY image of EVERY run

    # ---- device-resident timing (value)
    barrier()
    if sampler:
        sampler.mark_start()
    l0 = nat.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(args.steps):
        step_device(i)
    eng.post.sync()          # the last step's assembly + result copy run on the engine's second stream
    e1.record(stream)
    torch.cuda.synchronize()
    ms_dev = e0.elapsed_time(e1)
    launches = nat.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.fetch_arrays(check=False))
    barrier()

    # ---- end-to-end timing through the public API with host buffers (e2e): every step copies its uint8 frames from
    # pinned host memory and its results back; two runs are kept in flight (submit i+1, then read i), K results are read
    # inside the timed region.
    for i in range(4):          # pre-roll: both pinned host slots twice (staging buffers, plans and - small batches - graphs exist)
        fetch_e2e(submit_e2e(i))
    d2h_bytes.clear()
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    pending = submit_e2e(0)
    for i in range(1, args.steps):
        nxt = submit_e2e(i)
        fetch_e2e(pending)
        pending = nxt
    fetch_e2e(pending)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    barrier()

    status_bits = eng.post.status_accum()       # all images, warm-up excluded, both timed loops
    if world > 1:
        ms_dev = dist_mod.max_over_ranks(ms_dev, dev)
        ms_e2e = dist_mod.max_over_ranks(ms_e2e, dev)
        status_bits = int(dist_mod.max_over_ranks(status_bits, dev))     # bit set on any rank -> non-zero

    # ---- roofline of the dominant kernel (conv_tc_kernel), measured live: per-launch CUDA events, right after the timed
    # loops (same thermal / power state; the alternative workload below runs afterwards)
    roof = None
    if rank == 0 and not scales:      # (multi-scale: the plan held at the end is the last scale's, not a 368x368 forward)
        import ctypes
        step_device(0)
        torch.cuda.synchronize()
        cap = 64
        ms = (ctypes.c_float * cap)()
        fl = (ctypes.c_double * cap)()
        tot_ms, tot_fl, nl = 0.0, 0.0, 0
        for _ in range(3):
            nl = nat.lib().b200pose_net_profile(eng.net._h, ms, fl, cap, ctypes.c_void_p(sptr))
            if nl <= 0:
                break
            tot_ms += sum(ms[i] for i in range(1, nl))
            tot_fl += sum(fl[i] for i in range(1, nl))
        pk_tf, pk_bw, pk_src = peaks(clocks)
        if nl > 0 and tot_ms > 0:
            ach = tot_fl / (tot_ms * 1e-3) / 1e12
            first_ms = float(ms[0])                     # conv1_1 (CUDA-core launch) of the last profile pass
            net_ms = tot_ms / 3 + first_ms
            net_fl = tot_fl / 3 + fl[0]
            step_ms = ms_dev / args.steps
            roof = {"bound": "tensor", "kernel": "conv_tc_kernel (%d launches/step, all tcgen05 convs)" % (nl - 1),
                    "achieved": round(ach, 1), "peak": pk_tf, "unit": "TFLOP/s", "frac": round(ach / pk_tf, 4),
                    # DRAM bytes per launch cannot be read inside a timed run (it needs ncu's replay); the figure of the
                    # committed ncu capture of this command is in the file named below
                    "traffic": None,
                    "traffic_source": "profiles/r02_conv_tc_dram.csv (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch)",
                    "peak_source": pk_src,
                    "share_of_step": round(tot_ms / 3 / step_ms, 3),
                    # the same arithmetic over the whole network (conv1_1 included) and over the whole step
                    "net": {"achieved": round(net_fl / (net_ms * 1e-3) / 1e12, 1), "frac": round(net_fl / (net_ms * 1e-3) / 1e12 / pk_tf, 4),
                            "ms": round(net_ms, 4), "launches": nl},
                    "step": {"achieved": round(net_fl / (step_ms * 1e-3) / 1e12, 1),
                             "frac": round(net_fl / (step_ms * 1e-3) / 1e12 / pk_tf, 4), "ms": round(step_ms, 4)}}

    # ---- alternative workload: the same network pass per step, but the post-processing is fed person-like maps
    # (resident on the device) instead of the noise a random-weight network emits.  A trained model's maps look like
    # these; the number shows what the step costs when the post-processing is not the pathological case.
    alt = None
    if rank == 0 and not args.flip and not args.raw and not args.no_alt and not scales:
        import ctypes
        syn = importlib.import_module(_b200_alias.PKG + ".synthetic")
        heat, paf = syn.person_maps(BATCH, 8, seed=7)
        d_heat, d_paf = torch.from_numpy(heat).to(dev), torch.from_numpy(paf).to(dev)
        L = nat.lib()

        def step_alt(i):
            nat.check(L.b200pose_net_forward_u8(eng.net._h, ctypes.c_void_p(devin[i % n_rot].data_ptr()), 1, BATCH, H, W,
                                                eng.mode, None, 1, ctypes.c_void_p(sptr)), "b200pose_net_forward_u8")
            eng.post.run(d_heat.data_ptr(), d_paf.data_ptr(), True, 0, BATCH, H // 8, W // 8, 0.1, sptr)
        for i in range(3):
            step_alt(i)
        torch.cuda.synchronize()
        l_a = nat.launch_count()
        e0.record(stream)
        for i in range(args.steps):
            step_alt(i)
        eng.post.sync()
        e1.record(stream)
        torch.cuda.synchronize()
        ms_alt = e0.elapsed_time(e1)
        persons = sum(len(eng.post.humans(k)) for k in range(BATCH))
        alt = {"workload": "same network pass; post-processing on person-like maps resident on the device (8 schematic "
                           "persons per frame, synthetic.person_maps) instead of the random-weight network's noise maps",
               "value": round(BATCH * args.steps / (ms_alt * 1e-3), 2), "unit": UNIT,
               "ms_per_step": round(ms_alt / args.steps, 4), "persons_per_frame": round(persons / BATCH, 2),
               "gpu_launches": int(nat.launch_count() - l_a)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames = BATCH * world * args.steps
    value = frames / (ms_dev * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)
    cpu = cpu_baseline_sample(frames=2) if world == 1 and not args.no_cpu_baseline else None
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_dev / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"bf16": "bf16", "bf16x3": "bf16x3 (hi+lo bf16 planes, fp32 accumulate)", "fp32": "f32"}[args.mode],
        "data": "synthetic",
        "config": {"workload": "batch=%d per GPU, 368x368, rtpose VGG19 %s + fused NMS/PAF-match/assembly%s"
                               % (BATCH, {"bf16": "bf16 (tcgen05)", "bf16x3": "bf16x3 (tcgen05, split precision)", "fp32": "fp32 (CUDA cores, parity mode)"}[args.mode],
                                  (", multi-scale test-time averaging at scales %s%s (BASELINE.json configs[4]; %d forwards per frame; the "
                                   "composition has no reference counterpart: parity unpinned, DESIGN.md 2.7)"
                                   % (args.scales, " x left/right flip" if args.flip else "", len(scales) * (2 if args.flip else 1))) if scales else
                                  (" (BASELINE.json configs[2]; configs[3] when n_gpus=8)" if BATCH == 32 and not args.flip
                                   else (", left/right flip test-time averaging on the device (2 forwards per frame)" if args.flip else ""))),
                   "global_batch": BATCH * world, "weights": "He-normal seed 1234 (random init)",
                   "input": ("uint8 HWC BGR %dx%d frames, crop_with_factor (bilinear resize to 368x368) and rtpose_preprocess on "
                             "the device" % (SH, SW)) if args.raw else "uint8 HWC BGR frames, rtpose_preprocess fused on the device",
                   "l2": "inputs rotate over %d device batches (%d MB > 126 MB L2); ~%d MB of activations per step"
                         % (n_rot, n_rot * BATCH * SH * SW * 3 // 1000000, 44 * BATCH * (2 if args.flip else 1)),
                   "parallelism": "dp%d (frames sharded, one NCCL weight broadcast)" % world,
                   "post_status_bits": int(status_bits),
                   "post_status_scope": "OR over every image of every run of both timed loops (device-side accumulator)",
                   "workload_alt": alt},
        "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": BATCH * 3 * SH * SW * world,
                "d2h_bytes_per_step": (int(np.mean(d2h_bytes)) if d2h_bytes else 0) * world,   # rank 0's count x ranks
                "ms_per_step": round(ms_e2e / args.steps, 4)},
        "gpu_launches": int(launches) * world, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        "net_tflops_device": None if scales else round(FLOPS_PER_FRAME * (2 if args.flip else 1) * frames / (ms_dev * 1e-3) / 1e12 / world, 1),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def cpu_frame_fn():
    """The reference algorithm on the host: oracle port of rtpose_model.forward (torch CPU fp32) + NMS + the
    C pafprocess (oracle/_ref when it was built from the reference sources, else the plain-C port)."""
    import torch
    from oracle import glue_port, net_port, pafprocess_oracle
    sd = net_port.he_state_dict(1234)
    # "all the host threads it can use": torch's default is one thread per logical CPU; on many-core hosts the
    # conv stack is faster with fewer, so the best of {all, half, quarter} logical CPUs is used and reported.
    best = None
    probe = torch.rand((1, 3, H, W), generator=torch.Generator().manual_seed(1)) - 0.5
    for nt in sorted({os.cpu_count(), max(1, os.cpu_count() // 2), max(1, os.cpu_count() // 4)}, reverse=True):
        torch.set_num_threads(nt)
        with torch.no_grad():
            net_port.forward(sd, probe)
            t0 = time.perf_counter()
            net_port.forward(sd, probe)
            dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])
    cpu_frame_fn.threads = best[1]
    if pafprocess_oracle.have_ref():
        paf_lib, kind = pafprocess_oracle.load_ref(), "reference pafprocess.cpp + oracle port of the torch/numpy glue"
    else:
        paf_lib, kind = pafprocess_oracle.load_port(), "port"
    g = torch.Generator().manual_seed(1234)

    def one_frame():
        img = torch.randint(0, 256, (H, W, 3), generator=g, dtype=torch.uint8).numpy()
        x = torch.from_numpy(glue_port.rtpose_preprocess(img)[None])      # get_outputs minus imread (coco_eval.py:93-108)
        with torch.no_grad():
            (paf, heat), _ = net_port.forward(sd, x)
        heat = heat.numpy().transpose(0, 2, 3, 1)[0]
        paf = paf.numpy().transpose(0, 2, 3, 1)[0]
        return glue_port.paf_to_pose(heat, paf, paf_lib)      # paf_to_pose_cpp (paf_to_pose.py:372-406)
    return one_frame, kind


def cpu_baseline_sample(frames=2):
    one_frame, kind = cpu_frame_fn()
    one_frame()
    t0 = time.perf_counter()
    for _ in range(frames):
        one_frame()
    dt = time.perf_counter() - t0
    return {"value": round(frames / dt, 4), "unit": UNIT, "cores": getattr(cpu_frame_fn, "threads", os.cpu_count()),
            "kind": "port" if kind == "port" else "reference",
            "sample": "%d frames of 368x368, batch 1, serial run_eval-style loop (%s), after 1 warm-up frame" % (frames, kind)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    one_frame, kind = cpu_frame_fn()
    per_step = 1
    for _ in range(min(args.warmup, 1)):
        one_frame()
    t0 = time.perf_counter()
    for _ in range(args.steps * per_step):
        one_frame()
    dt = time.perf_counter() - t0
    v = args.steps * per_step / dt
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": round(dt / args.steps * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "batch=32 per GPU, 368x368, rtpose VGG19 + pafprocess; each step = a bounded sample "
                                   "of %d frame(s) run serially at batch 1 on the host CPU" % per_step},
            "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": getattr(cpu_frame_fn, "threads", os.cpu_count()),
                             "kind": "port" if kind == "port" else "reference",
                             "sample": "%d frame(s) per step, %d steps (%s)" % (per_step, args.steps, kind)},
            "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="bf16", choices=["bf16", "bf16x3", "fp32"],
                    help="arithmetic of the network (the headline config is bf16; bf16x3 / fp32 price the tighter tolerances)")
    ap.add_argument("--no-alt", action="store_true", help="skip the person-like-maps alternative workload")
    ap.add_argument("--batch", type=int, default=32, help="frames per GPU per step (the headline config is 32)")
    ap.add_argument("--flip", action="store_true", help="left/right flip test-time averaging (2 forwards per frame)")
    ap.add_argument("--scales", default="", metavar="S1,S2,...",
                    help="multi-scale test-time averaging around 368 (BASELINE.json configs[4]: 0.5,1.0,1.5,2.0 with --flip --batch 8)")
    ap.add_argument("--raw", type=int, default=0, metavar="N",
                    help="feed N x N raw frames and run crop_with_factor (resize to 368 x 368) on the device as well")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the persons the last step found (rank 0) to DIR/*.npy; the inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3)
    global BATCH
    BATCH = args.batch
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
