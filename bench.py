#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 visualDet3D hot path (contract: see the task brief / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config stereo|gac|monoflex|km3d|yolo3d] [--batch B]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, NCCL)

Default workload (= BASELINE.json configs[1] / the `metric`): a "step" = one YOLOStereo3D forward (backbone -> cost volumes -> neck ->
head -> decode -> NMS) over a batch of 8 synthetic 384x1280 stereo pairs per GPU; ranks hold disjoint pairs (weak scaling) and exchange
only one all-gather of detection records per step.  `--config` selects the other BASELINE configs (gac = configs[2] with the yaw
post-optimisation of its shipped config on, monoflex / km3d = configs[3], yolo3d = configs[0] on the GPU).  Prints ONE JSON line on rank 0.

  value        whole-job samples/s, inputs resident in HBM, CUDA events, max over ranks; the record all-gather of every step is inside
               the timed region (on a side stream, one step behind the compute stream)
  e2e          same metric through the public pipeline API with HOST buffers: pinned uint8 camera frames -> H2D -> device input pipeline
               (crop / resize / normalise) -> forward -> all-gather -> D2H of the records; `e2e_f32` = the same with float32 network
               inputs (4x the H2D bytes), the form round 1 reported
  roofline     scale-4 PSMCosine kernel (dominant cost-volume kernel; stereo only): algorithmic bytes / CUDA-event time vs measured HBM peak
  --dump-outputs DIR : after the timing, DIR/<name>.npy holds what the last timed step of each leg returned (per-image scores, boxes,
               classes and detection counts; the device leg's record block too): inputs and weights are seeded, so two builds of the project
               can be compared output for output
  cpu_baseline / --impl reference : the UNMODIFIED reference (a checkout found by oracle/refload.py, e.g. via $VISUALDET3D_REF)
               running its own PyTorch forward on this host's cores (`kind: "reference"`); falls back to the oracle port (`"port"`)
               when no reference checkout is importable on this machine
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (metric, unit, H, W, default batch, workload text)
    "stereo": ("synthetic_384x1280_stereo_pairs_per_sec", "pairs/s", 384, 1280, 8, "YOLOStereo3D forward, batch {B} stereo 384x1280 per GPU, ResNet-34"),
    "gac": ("synthetic_288x1280_mono_images_per_sec", "images/s", 288, 1280, 8,
            "GroundAwareYolo3D (GAC head, ResNet-101) forward, batch {B} mono 288x1280 per GPU, post_optimization on"),
    "monoflex": ("synthetic_384x1280_mono_images_per_sec", "images/s", 384, 1280, 8, "MonoFlex (DLA-34 + 16 DCNv2) forward, batch {B} mono 384x1280 per GPU"),
    "km3d": ("synthetic_384x1280_mono_images_per_sec", "images/s", 384, 1280, 8, "KM3D (DLA-34 + 16 DCNv2) forward, batch {B} mono 384x1280 per GPU"),
    "yolo3d": ("synthetic_288x1280_mono_images_per_sec", "images/s", 288, 1280, 1, "Yolo3D (ResNet-18, DCNv2 head) forward, batch {B} mono 288x1280 per GPU"),
}
FRAME_HW = (375, 1242)                                           # a KITTI camera frame; crop_top below gives the network aspect ratio
PSM4_NCU_TRAFFIC_B8 = 137_400_000                                # DRAM bytes per launch of the scale-4 PSMCosine kernel at B = 8 (ncu)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock / power / throttle-reason sampling DURING the timed region (B200_PROFILING.md): NVML polled every 5 ms from a
    thread (nvidia_ml_py), falling back to `nvidia-smi -lms` when NVML is not importable."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.h, self.stop_flag, self.samples = None, None, False, []
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(physical_index(index))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(self.h) / 1e3
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nvml is not None:
            self.stop_flag, self.samples = False, []
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={physical_index(self.index)}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            n = self.nvml
            try:
                mx = float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM))
            except Exception:
                mx = None
            sm = [float(a) for a, _, _ in self.samples]
            pw = [b for _, b, _ in self.samples]
            bits = 0
            for _, _, r in self.samples:
                bits |= int(r)
            reasons = sorted(k for k, v in self.BITS.items() if bits & v)
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": mx,
                    "power_w": statistics.median(pw) if pw else None, "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def physical_index(local_index: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis and all(v.strip().isdigit() for v in vis.split(",")) and local_index < len(vis.split(",")):
        return int(vis.split(",")[local_index])
    return local_index


def bind_to_gpu_numa_node(local_index: int):
    """Pin this rank's host threads to the CPU cores NVML reports as local to its GPU, BEFORE any pinned buffer is allocated (first
    touch then places the staging buffers on the GPU's NUMA node).  Returns the number of cores bound to, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(physical_index(local_index))
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i * 64 + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# =====================================================================================================================
# reference arm: the reference's own CPU forward (the real package when it is on this box, else the oracle port)
# =====================================================================================================================
def _usable_cpus() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _reference_callable(config: str):
    """-> (kind, fn) with fn() = one forward of ONE sample (pair / image) at the config's full resolution on the host."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refload
    from visualdet3d_b200 import synth
    _, _, H, W, _, _ = CONFIGS[config]
    if config == "stereo":
        from visualdet3d_b200.detectors import build_synthetic_stereo3d
        det, sd, cfg, (pm, ps) = build_synthetic_stereo3d(seed=0)
        left, right, P2, P3 = synth.synth_stereo_inputs(1, H, W, seed=1)
        inputs = [left, right, P2, P3]
        name = "Stereo3D"
    else:
        from visualdet3d_b200.detectors import build_synthetic_mono3d, build_synthetic_monoflex
        name = {"gac": "GroundAwareYolo3D", "yolo3d": "Yolo3D", "monoflex": "MonoFlex", "km3d": "KM3D"}[config]
        if config in ("gac", "yolo3d"):
            det, sd, cfg, (pm, ps) = build_synthetic_mono3d(name, seed=0)
        else:
            det, sd, cfg = build_synthetic_monoflex(seed=0, name=name)
            pm = ps = None
        img, P2 = synth.synth_mono_inputs(1, H, W, seed=1)
        inputs = [img, P2]
    if refload.available():
        refload.load_reference()                       # CPU mode: the unmodified reference, `.cuda()` calls are no-ops
        from visualDet3D.networks.utils.registry import DETECTOR_DICT
        model = DETECTOR_DICT[name](refload.to_edict(cfg))
        model.load_state_dict(sd, strict=False)
        model.eval()

        import contextlib

        def fn():
            with torch.no_grad(), contextlib.redirect_stdout(open(os.devnull, "w")):     # the reference's @profile decorators print timings
                return model(list(inputs))
        return "reference", fn
    import torch_port as tp

    def fn_port():
        if config == "stereo":
            return tp.stereo3d_forward(sd, inputs[0], inputs[1], inputs[2], cfg, pm, ps)
        if config in ("gac", "yolo3d"):
            return tp.mono3d_forward(sd, inputs[0], inputs[1], cfg, pm, ps)
        return (tp.km3d_forward if config == "km3d" else tp.monoflex_forward)(sd, inputs[0], inputs[1], cfg)
    return "port", fn_port


def pick_cpu_threads(fn):
    """Thread count for the CPU arm, calibrated ON THE WORKLOAD ITSELF: one warm forward + one timed forward per candidate
    (8, 16, 32, 64, all usable cores), fastest wins.  `torch.set_num_threads(nproc = 128)` is pathologically slow for oneDNN convs on
    the GPU boxes (28 s per pair), so "all cores" is a candidate, not the rule; the chosen count is what `cores` reports."""
    import torch
    avail = _usable_cpus()
    best, best_t, tried = None, None, {}
    for n in sorted({c for c in (8, 16, 32, 64, avail) if c <= avail}):
        torch.set_num_threads(n)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        tried[n] = round(dt, 3)
        if best_t is None or dt < best_t:
            best, best_t = n, dt
        if dt > 20.0:                # a pathological setting: do not spend more of the sample budget on larger counts
            break
    torch.set_num_threads(best)
    return best, tried


def run_reference(args):
    """--impl reference: the reference's own CPU forward on this box's host cores, on the arm's config / metric / unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    metric, unit, H, W, defB, text = CONFIGS[args.config]
    B = args.batch or defB
    kind, fn = _reference_callable(args.config)
    cores, tried = pick_cpu_threads(fn)
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        fn()
    steps = max(1, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    dt = time.perf_counter() - t0
    v = steps / dt
    sample = (f"{steps} forwards of 1 sample at {H}x{W} = a bounded sample of the batch-{B} step (the reference asserts batch 1: "
              f"yolostereo3d_detector.py:78); {kind} on {cores} of {_usable_cpus()} usable host threads (per-candidate seconds: {tried})")
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": text.format(B=B) + f" (CPU arm: {sample})"},
        "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_subprocess(config: str, batch: int):
    """The CPU arm in its own process (importing the reference patches torch globally): 3 timed forwards."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", config, "--batch", str(batch),
                            "--steps", "3", "--warmup", "1"], capture_output=True, text=True, timeout=900,
                           env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)["cpu_baseline"]
    except Exception as e:            # the GPU numbers stand on their own; say why the baseline is missing
        return {"value": None, "unit": CONFIGS[config][1], "cores": None, "kind": "unavailable", "sample": f"CPU arm failed: {e!r}"[:300]}


# =====================================================================================================================
def build_detector(config: str):
    from visualdet3d_b200.detectors import build_synthetic_mono3d, build_synthetic_monoflex, build_synthetic_stereo3d
    if config == "stereo":
        return build_synthetic_stereo3d(seed=0)[0]
    if config == "gac":
        det = build_synthetic_mono3d("GroundAwareYolo3D", seed=0)[0]
        det.post_optimization = True          # R/config/Yolo3D_example: head.test_cfg.post_optimization = True
        return det
    if config == "yolo3d":
        return build_synthetic_mono3d("Yolo3D", seed=0, depth=18)[0]
    return build_synthetic_monoflex(seed=0, name={"monoflex": "MonoFlex", "km3d": "KM3D"}[config])[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="stereo", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="samples per GPU per step (default: 8; yolo3d 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-mode", action="store_true", help="device-resident steps only (for ncu): no e2e leg, no CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of every leg to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.profile_mode or args.impl == "reference"):
        ap.error("--dump-outputs writes the outputs of the timed B200 legs: not with --profile-mode or --impl reference")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    numa_cores = bind_to_gpu_numa_node(local_rank) if world > 1 else None

    import torch
    import torch.distributed as dist
    from visualdet3d_b200 import _lib, synth, parallel
    from visualdet3d_b200.pipeline import StreamedInference

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: the "NCCL version ..." banner the library prints to stdout when the first communicator is created
        # is sent to stderr instead (file-descriptor level: the print comes from C code)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    warmup_requested = args.warmup
    args.warmup = max(args.warmup, 4)            # >= 3 by contract; 4 so that both record buffers have had their eager step and their graph capture
    metric, unit, H, W, defB, text = CONFIGS[args.config]
    B = args.batch or defB
    kmax = 512
    stereo = args.config == "stereo"
    n_img = 2 if stereo else 1

    det = build_detector(args.config).to(dev).eval()

    def make_inputs(seed):
        """every rank owns its own B samples of the global batch (weak scaling): a different seed per rank"""
        if stereo:
            l, r, p2, _ = synth.synth_stereo_inputs(B, H, W, seed=seed)
            return [l, r], p2
        im, p2 = synth.synth_mono_inputs(B, H, W, seed=seed)
        return [im], p2

    imgs, P2 = make_inputs(1 + rank)
    h_imgs, h_p2 = [t.pin_memory() for t in imgs], P2.pin_memory()
    d_imgs, d_p2 = [t.to(dev) for t in h_imgs], h_p2.to(dev)
    # uint8 camera frames for the headline e2e leg: crop_top chosen so that (Hf - crop) / Wf matches the network aspect as the reference's
    # CropTop + Resize do (R/data/pipeline/stereo_augmentator.py:63-134,213-258); the resized frame is zero-padded on the right to W
    Hf, Wf = FRAME_HW
    crop_top = max(0, Hf - int(round(Wf * H / W)))
    g = torch.Generator().manual_seed(100 + rank)
    h_frames = [torch.randint(0, 256, (B, Hf, Wf, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(n_img)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    side = torch.cuda.Stream(device=dev) if world > 1 else None
    rec_bufs = [torch.empty(B, 1 + kmax * parallel.REC, device=dev) for _ in range(2)]
    gat_bufs = [torch.empty(world * B, 1 + kmax * parallel.REC, device=dev) for _ in range(2)] if world > 1 else None
    ev_pack = [torch.cuda.Event() for _ in range(2)]
    ev_gath = [torch.cuda.Event() for _ in range(2)]

    from visualdet3d_b200.graphs import GraphedStep
    use_graphs = os.environ.get("VD3D_GRAPHS", "1") != "0" and not args.profile_mode      # (ncu launch lists are taken from eager launches)
    steps = [GraphedStep(det, d_imgs, d_p2, rec_bufs[k], kmax, enabled=use_graphs) for k in range(2)]

    def graph_launches():
        return sum(s.replays * s.launches_per_replay for s in steps) + sum(s.replays * s.launches_per_replay for s in pipe._steps.values())

    def step_device(i):
        """one device-resident step: forward .. NMS (+ post-optimisation) -> record block -> all-gather (side stream, overlapping the next
        step's forward; buffer i % 2 is reused only after its previous gather has completed)"""
        k = i % 2
        cur = torch.cuda.current_stream()
        if world > 1 and i >= 2:
            cur.wait_event(ev_gath[k])
        dec = steps[k]()                          # forward .. NMS (+ post-optimisation) + record block: eager, then one CUDA graph per buffer
        rec = rec_bufs[k]
        if world > 1:
            ev_pack[k].record(cur)
            with torch.cuda.stream(side):
                side.wait_event(ev_pack[k])
                parallel.all_gather_records(rec, out=gat_bufs[k])
                ev_gath[k].record(side)
        return dec, rec

    def drain():
        if world > 1:
            torch.cuda.current_stream().wait_stream(side)

    pipe = StreamedInference(det, B, H, W, kmax=kmax, world=world, frame_hw=(Hf, Wf), crop_top=crop_top, graphs=use_graphs)

    def run_e2e(nsteps, frames: bool):
        """`nsteps` batches through the public host-fed pipeline: every batch pays its pinned-host -> device copy and the
        device -> host read of the gathered detection records; copy of batch i+1 overlaps the forward of batch i."""
        out = prev = None
        for _ in range(nsteps):
            t = pipe.submit_frames(*h_frames, h_p2) if frames else pipe.submit(*h_imgs, h_p2)
            if prev is not None:
                out = pipe.collect(prev)
            prev = t
        out = pipe.collect(prev)
        return out

    with torch.no_grad():
        for i in range(args.warmup):
            step_device(i)
            drain()
            if not args.profile_mode:
                run_e2e(1, True)
                run_e2e(1, False)
        if args.profile_mode:
            torch.cuda.synchronize()
            _lib.launch_count_reset()
            for i in range(args.steps):
                step_device(i)
            drain()
            torch.cuda.synchronize()
            print(json.dumps({"profile_mode": True, "config": args.config, "launches_per_step": _lib.launch_count() / args.steps}))
            return
        # ---------------- device-resident timing ----------------------------------------------------------------
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        det.profile_events = [] if stereo else None
        _lib.launch_count_reset()
        g0 = graph_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        e_fwd = torch.cuda.Event(enable_timing=True)
        for i in range(args.steps):
            step_device(i)
        e_fwd.record()                            # this rank's own forwards are done (per_rank.forward_ms_per_step: shows a slow GPU)
        drain()                                   # the last all-gathers are inside the timed region
        e1.record()
        barrier()
        last_records = (gat_bufs if world > 1 else rec_bufs)[(args.steps - 1) % 2].clone()     # the last timed step's (gathered) records
        launches = _lib.launch_count() + graph_launches() - g0          # kernels launched directly + kernels inside the replayed graphs
        ms_dev = e0.elapsed_time(e1)
        ms_fwd = e0.elapsed_time(e_fwd)
        situ = {}
        if stereo:
            for nm, a, b in det.profile_events:
                situ.setdefault(nm, []).append(a.elapsed_time(b))
        psm_ms = situ.get("psm4", [])
        det.profile_events = None
        clocks = sampler.stop()
        if E_overflow():
            raise SystemExit("bench.py: fp16-range guard tripped during the timed region")

        # ---------------- end-to-end timing (host inputs): uint8 frames (headline) and float32 inputs ---------------------
        def time_e2e(frames):
            barrier()
            t0 = time.perf_counter()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            res = run_e2e(args.steps, frames)
            b.record()
            barrier()
            return max(a.elapsed_time(b), 1e3 * (time.perf_counter() - t0)), res      # device time and host wall clock: the larger one
        ms_e2e, res_u8 = time_e2e(True)
        ms_e2e_f32, res_f32 = time_e2e(False)
        # ---------------- multi-GPU correctness on hardware --------------------------------------------------------
        gather_verified = None
        if world > 1:
            dec, rec = step_device(0)
            drain()
            torch.cuda.synchronize()
            gathered = gat_bufs[0]
            ok = torch.equal(gathered[rank * B:(rank + 1) * B], rec)                 # my slice of the gathered block == my local block, bit for bit
            if rank == 0:                                                             # rank 0 recomputes every other rank's batch itself
                for r in range(1, world):
                    im_r, p2_r = make_inputs(1 + r)
                    dec_r = det.launch(*[t.to(dev) for t in im_r], p2_r.to(dev))
                    rec_r = parallel.pack_records_device(dec_r, kmax)
                    torch.cuda.synchronize()
                    ok = ok and torch.equal(gathered[r * B:(r + 1) * B], rec_r)
            flag = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            gather_verified = bool(flag.item())
    t = torch.tensor([ms_dev, ms_e2e, ms_e2e_f32], device=dev, dtype=torch.float64)
    per_rank = None
    if world > 1:
        mine = {"rank": rank, "ms_per_step": ms_dev / args.steps, "forward_ms_per_step": ms_fwd / args.steps, "e2e_ms_per_step": ms_e2e / args.steps, "sm_mhz": clocks.get("sm_mhz"),
                "sm_min_mhz": clocks.get("sm_min_mhz"), "power_w": clocks.get("power_w"), "reasons": clocks.get("reasons"), "numa_cores": numa_cores}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_e2e_f32 = t.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total = B * world * args.steps
    value = total / (ms_dev / 1e3)
    peak, peak_kind = measured_peaks()
    out = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": warmup_requested,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": text.format(B=B) + ", random-init seeded weights", "name": args.config,
                   "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2": "activations + weights of one step exceed the 126 MB L2 several times over; no explicit flush",
                   "warmup_steps_run": args.warmup,
                   "conv_engine": os.environ.get("VD3D_CONV_ENGINE", "default"),
                   "cuda_graphs": ("one graph per record buffer / staging slot (graphs.GraphedStep); the stereo device-resident leg stays eager for the "
                                   "in-situ event timing of its cost-volume kernels" if use_graphs else "off"),
                   "detections_per_step": sum(len(r[0]) for r in res_f32[rank * B:(rank + 1) * B]),
                   "all_gather": "one all_gather_into_tensor of the record block per step, on a side stream one step behind the forward"},
        "e2e": {"value": total / (ms_e2e / 1e3), "unit": unit, "h2d_bytes_per_step": int(pipe.h2d_bytes_frames), "d2h_bytes_per_step": int(pipe.d2h_bytes),
                "ms_per_step": ms_e2e / args.steps, "input": f"pinned uint8 camera frames {Hf}x{Wf}x3 (crop_top {crop_top}) -> device crop / resize / normalise",
                "api": "visualdet3d_b200.pipeline.StreamedInference.submit_frames / collect (double-buffered H2D on a copy stream, async D2H of the gathered records)"},
        "e2e_f32": {"value": total / (ms_e2e_f32 / 1e3), "unit": unit, "h2d_bytes_per_step": int(pipe.h2d_bytes), "d2h_bytes_per_step": int(pipe.d2h_bytes),
                    "ms_per_step": ms_e2e_f32 / args.steps, "input": "pinned float32 network inputs", "api": "StreamedInference.submit / collect"},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if world > 1:
        out["gather_verified"] = gather_verified
        out["per_rank"] = per_rank
    if stereo:
        psm_bytes = 4 * (H // 4) * (W // 4) * (2 * 64 + 24) * B                  # SURVEY.md 8(d): 18,677,760 B per pair
        psm_avg_ms = statistics.mean(psm_ms) if psm_ms else None
        achieved = (psm_bytes / 1e9) / (psm_avg_ms / 1e3) if psm_avg_ms else None
        tc = os.environ.get("VD3D_PSM_ENGINE", "tc") == "tc" and os.environ.get("VD3D_CONV_ENGINE", "tc16") == "tc16"
        out["roofline"] = {"kernel": "psm_cosine_tc_kernel (scale-4 PSMCosine, tcgen05 on fp16 hi/lo planes)" if tc
                           else "psm_cosine_nhwc_v4_kernel<64> (scale-4 PSMCosine, SIMT)",
                           "bound": "hbm", "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                           "frac": (achieved / peak) if achieved else None, "avg_launch_ms": psm_avg_ms, "algorithmic_bytes_per_launch": psm_bytes,
                           # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at B = 8 from the committed `ncu --set full` capture
                           "traffic": (PSM4_NCU_TRAFFIC_B8 if (B == 8 and tc) else None),
                           "traffic_source": "ncu --set full, one launch, profiles/r01_ncu_psm_cosine_tc.txt (round 2 re-capture, profiles/r02_ncu_misc.txt row 10: 125.9 MB read + 11.3 MB written)"}
        # the other cost-volume kernels, timed in situ the same way (SURVEY.md 8(d) algorithmic bytes per pair x batch)
        alg = {"psm8": 4 * (H // 8) * (W // 8) * (2 * 128 + 24) * B, "concat_volume": (2 * 8 * (H // 16) * (W // 16) * 4 + 16 * 12 * (H // 16) * (W // 16) * 4) * B}
        out["cost_volume_in_situ"] = {k: {"avg_launch_ms": statistics.mean(v), "algorithmic_bytes": alg[k], "GB_per_s": alg[k] / 1e9 / (statistics.mean(v) / 1e3),
                                          "frac_of_hbm_peak": alg[k] / 1e9 / (statistics.mean(v) / 1e3) / peak} for k, v in situ.items() if k in alg and v}
    if not args.no_cpu_baseline and world == 1:          # the CPU arm is timed on rank 0 at N = 1 only (the driver runs --impl reference for every N)
        out["cpu_baseline"] = cpu_baseline_subprocess(args.config, B)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"device": parallel.unpack_records(last_records.cpu()), "e2e": res_u8, "e2e_f32": res_f32}, last_records)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(dirname: str, legs, records) -> None:
    """legs: leg name -> per-image (scores, boxes, classes) of the GLOBAL batch; records: the device leg's record block."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    arrays = {"device_records": records.cpu()}
    for leg, res in legs.items():
        arrays[f"{leg}_counts"] = torch.tensor([len(s) for s, _, _ in res])
        for i, what in enumerate(("scores", "boxes", "classes")):
            arrays[f"{leg}_{what}"] = torch.cat([r[i].cpu() for r in res])
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a.to(torch.float32).numpy())


def E_overflow() -> bool:
    from visualdet3d_b200 import engine
    return engine.fp16_range_overflowed()


if __name__ == "__main__":
    main()
