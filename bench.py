#!/usr/bin/env python
"""bench.py -- VIO frames/sec of the R-VIO hot path (tracker + MSCKF update) on B200, and the CPU reference arm.

Contract (see task statement): `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line.
  step      = one frame of the hot path on a seeded synthetic EuRoC-shaped stream (BASELINE.json configs[1] by default:
              752x480 mono + 200 Hz IMU, 200 features, 11-clone window), i.e. one System::MonoVIO iteration, the corner detector
              (FeatureDetector::DetectWithSubPix) included in every step of both arms (--detector inloop, the default).
  value     = frames/s with the frames already resident in HBM (rvio_vio_step_dev).
  e2e       = frames/s through the public C ABI with HOST buffers in pinned memory: per timed step one frame upload (frame k+1,
              announced while frame k is processed: rvio_vio_prefetch), the IMU rows up, the pose back; e2e.strict = the same
              without the announcement (every step uploads its own frame before its first kernel can start).
  roofline  = dominant kernel of a step's critical path (per-kernel CUDA events recorded by the library on its own stream).
  cpu_baseline / --impl reference = the same loop on the host cores: OpenCV stages through the real OpenCV (cv2, all
              threads), Eigen stages through the single-threaded C restatement in oracle/ (the reference is single threaded).
Order of a run: untimed settling passes, the three measured legs (e2e.strict, e2e, value), their reduction over the ranks, then the
extra legs under a deadline (stage timeline, per-kernel profile, 8 streams per GPU, N > 1: the configs[4] stream feature-sharded
over the N GPUs, N = 1: configs[2] stream, worst-case updates, CPU baseline).
N > 1: one process per GPU, each rank runs an independent stream (BASELINE configs[3] style replicas, no collective on the
data path); value = total frames / max-over-ranks time ("scaling": "weak").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20260922
T_STATIC = 0.5
# Seed of the configs[4] stream of the `sharded` leg.  The reference's motion detector (System.cc:203-214: 0.005 rad or 1 cm inside ONE
# frame interval) fires late on these gently ramped trajectories, and the filter then starts from "at rest" with whatever velocity the
# trajectory already has; with SEED + 4 that is 1.1 m/s at frame 28: the filter never recovers, LM / the gate reject every track (in the
# CPU oracle alike) and the update is a pass-through.  20260953 is detected at frame 20 with 0.07 m/s: every track is accepted and the
# window-full frames carry 500-1000 features (stacked H up to 60 000 x 180) -- the update the sharding is meant for.
SHARDED_SEED = 20260953


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, help="BASELINE.json configs index (1 = headline)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the feature-sharded configs[4] leg (N > 1 only)")
    ap.add_argument("--no-extra-legs", action="store_true", help="skip the configs[2] stress stream and the worst-case update micro-benchmarks")
    ap.add_argument("--detector", default="inloop", choices=["inloop", "precomputed"],
                    help="inloop (default): FeatureDetector::DetectWithSubPix runs inside every timed step, on the GPU in this arm and "
                         "through cv2 in the reference arm (the whole Tracker::track); precomputed: corner candidates prepared "
                         "beforehand, identical for both arms")
    ap.add_argument("--batch-streams", type=int, default=8, help="extra leg: independent streams run concurrently on one GPU (BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of the device-resident leg returned as DIR/<name>.npy "
                         "(float64): pose, state_x, state_P, update_info; the inputs are seeded, so two builds can be compared output "
                         "for output (rank 0 only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


# ----------------------------------------------------------------------------------------- workload
def make_workload(cfg, n_frames, seed, precompute=True):
    """Seeded stream + per-frame IMU slices + corner candidates (s=1 and s=2 spacing) from the equalised frames."""
    import cv2
    import rvio_b200  # noqa: F401
    from rvio_b200 import synth
    st = synth.Stream(cfg, n_frames, seed, t_static=T_STATIC)
    consumed = 0
    imus = []
    for i in range(n_frames):
        imu, consumed = st.imu_for_frame(i, consumed)
        imus.append(np.ascontiguousarray(imu))
    clahe = cv2.createCLAHE(3.0, (5, 5))
    cand1, cand2, eqs = [], [], []
    q = float(np.float32(cfg.qual_lvl)); md = float(np.float32(cfg.min_dist))
    for f in st.frames:
        if not precompute:                                 # the detector runs inside the timed step
            cand1.append(np.zeros((0, 2), np.float32)); cand2.append(np.zeros((0, 2), np.float32))
            continue
        eq = clahe.apply(f) if cfg.enable_equalizer else f
        eqs.append(eq)
        c1 = cv2.goodFeaturesToTrack(eq, cfg.n_features, q, md)
        c2 = cv2.goodFeaturesToTrack(eq, cfg.n_features, q, 2 * md)
        cand1.append(np.zeros((0, 2), np.float32) if c1 is None else np.ascontiguousarray(c1.reshape(-1, 2), np.float32))
        cand2.append(np.zeros((0, 2), np.float32) if c2 is None else np.ascontiguousarray(c2.reshape(-1, 2), np.float32))
    return dict(stream=st, frames=st.frames, imus=imus, cand1=cand1, cand2=cand2, eqs=eqs)


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region, read in-process through NVML (nvidia-ml-py) every 100 ms: no
    nvidia-smi process is forked while a step is being timed (round 1 forked one per rank every 200 ms).  Falls back to one
    nvidia-smi query before and one after the region when NVML cannot be loaded."""
    _BITS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.samples, self.max_mhz, self.reasons, self.power = [], None, set(), []
        self.stop = False
        self.index = index
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
        self.th = threading.Thread(target=self.run, daemon=True)

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:
                return index
        return index

    def _nvml_sample(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
        except Exception:
            pass
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in self._BITS.items():
            if r & bit:
                self.reasons.add(name)

    def _smi_sample(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip().split(",")
            self.samples.append(float(out[0])); self.max_mhz = float(out[1])
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                if "Active" in val and "Not" not in val:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self.stop:
            try:
                self._nvml_sample()
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        if self.nv is not None:
            self.th.start()
        else:
            self._smi_sample()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.nv is not None:
            self.th.join(timeout=3)
        else:
            self._smi_sample()

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": max(self.power) if self.power else None,
                "how": "NVML in-process, 100 ms" if self.nv is not None else "nvidia-smi before/after the timed region"}


def bind_to_gpu_numa_node(local_rank):
    """Pins this rank (and the pinned staging buffers it allocates afterwards, by first touch) to the CPUs of the NUMA node
    its GPU hangs off, split evenly between the ranks that share the node.  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(ClockSampler._physical_index(local_rank))
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        path = f"/sys/bus/pci/devices/{bus}/"
        node = int(open(path + "numa_node").read())
        cpus = open(path + "local_cpulist").read().strip()
        ids = []
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.extend(range(int(a), int(b or a) + 1))
        ids = sorted(set(ids) & os.sched_getaffinity(0))
        if not ids:
            return {"numa_node": node, "bound": False}
        # ranks on the same node take disjoint slices
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        per_node = max(1, (local_world + 1) // 2) if local_world > 1 else 1
        k = local_rank % per_node
        sl = ids[k * len(ids) // per_node:(k + 1) * len(ids) // per_node] or ids
        os.sched_setaffinity(0, sl)
        return {"numa_node": node, "bound": True, "cpus": f"{sl[0]}-{sl[-1]} ({len(sl)})"}
    except Exception as e:          # pragma: no cover
        return {"bound": False, "why": repr(e)[:80]}


# ----------------------------------------------------------------------------------------- B200 arm
_LAST_DRIVE = {}
_LAST_POSE = {}
_RAW = {}


def raw_abi(L):
    """The four per-frame entry points with plain-pointer prototypes (what a C / C++ host hands to the C ABI): the timed loop passes
    addresses computed beforehand instead of going through the NumPy-checking Python adaptor (r-vio_b200/host.py: ~15 us per step of
    ndpointer validation and array normalisation that a compiled host does not have)."""
    import ctypes as C
    if not _RAW:
        vp, ci = C.c_void_p, C.c_int
        for name, args in (("rvio_vio_step", [vp, vp, ci, ci, ci, ci, vp, ci, vp, ci, ci, vp, vp]),
                           ("rvio_vio_step_dev", [vp, vp, ci, vp, ci, vp, ci, ci, vp, vp]),
                           ("rvio_vio_prefetch", [vp, vp, ci, ci, ci, ci]),
                           ("rvio_vio_prefetch_fence", [vp, vp])):
            f = L[name]                                    # a fresh function object: the adaptor's own prototypes stay as they are
            f.argtypes = args
            f.restype = ci
            _RAW[name] = f
    return _RAW


def drive(L, vio, wl, K, W, dev, inloop, dev_inputs, flush, prefetch=False):
    """pre-roll until the first valid pose, W warm-up steps, K timed steps (per-step CUDA events on the library's own stream,
    L2 flush between timed steps outside the event pair).  Returns (per-step ms list, wall seconds, launches, frames used)."""
    import torch
    frames, imus = wl["frames"], wl["imus"]
    n_frames = len(frames)
    stream = torch.cuda.ExternalStream(L.rvio_tracker_stream(L.rvio_vio_tracker(vio.h)), device=dev)
    if not dev_inputs:
        # e2e leg: host frames in PINNED memory (the contract's "host->device copy of that step's inputs from pinned host
        # memory"); the library DMA's a pinned single-channel frame straight into its gray buffer inside the timed call
        keep = [torch.from_numpy(f).pin_memory() for f in frames]
        frames = [k.numpy() for k in keep]
    if dev_inputs:
        d_frames = [torch.from_numpy(f).to(dev) for f in frames]
        d_c1 = [torch.from_numpy(c).to(dev) if len(c) else None for c in wl["cand1"]]
        d_c2 = [torch.from_numpy(c).to(dev) if len(c) else None for c in wl["cand2"]]
        torch.cuda.synchronize()
    # ---- everything the per-frame calls need, as plain addresses (device detector mode; the precomputed-candidates protocol keeps the
    #      Python adaptor)
    import ctypes as C
    from rvio_b200 import capi
    raw = raw_abi(L) if inloop else None
    if raw:
        Wpx, Hpx = int(frames[0].shape[1]), int(frames[0].shape[0])
        imu_ptr = [int(a.ctypes.data) for a in imus]
        imu_n = [int(a.shape[0]) for a in imus]
        assert all(a.dtype == np.float64 and a.flags.c_contiguous and (a.ndim == 2 and a.shape[1] == 8 or a.size == 0) for a in imus)
        if dev_inputs:
            img_ptr = [int(t.data_ptr()) for t in d_frames]
        else:
            assert all(f.dtype == np.uint8 and f.flags.c_contiguous and f.shape == (Hpx, Wpx) for f in frames)
            img_ptr = [int(f.ctypes.data) for f in frames]
        pose_buf = np.zeros(7); pose_ptr = int(pose_buf.ctypes.data)
        valid = C.c_int(0); valid_ptr = C.addressof(valid)
        r_step, r_step_dev, r_pref, r_fence = (raw["rvio_vio_step"], raw["rvio_vio_step_dev"], raw["rvio_vio_prefetch"],
                                               raw["rvio_vio_prefetch_fence"])
        hnd = vio.h
    got_pose = False
    i = 0
    timed, warm = 0, 0
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    launches0 = None
    wall = 0.0
    infos = []
    host_tl = np.zeros(8, np.float32); host_us = []
    stage_diag = bool(os.environ.get("RVIO_BENCH_STAGES_IN_LEGS"))        # diagnostic: stage stamps inside the measured legs (adds ~7 us / step)
    if stage_diag:
        L.rvio_vio_timeline(vio.h, 1, None)
    stages = []
    while timed < K:
        if i >= n_frames:
            raise RuntimeError("stream too short for the requested steps")
        cands = wl["cand2"] if got_pose else wl["cand1"]
        timing = got_pose and warm >= W
        if timing:
            if not os.environ.get("RVIO_BENCH_NO_FLUSH"):              # diagnostic switch only: a number taken without the flush is not a bench value
                flush.fill_(timed & 0xff)                              # L2 flush between timed iterations (untimed)
            torch.cuda.synchronize()
            if launches0 is None:
                launches0 = L.rvio_b200_kernel_launches()
            ev0[timed].record(stream)
            t0 = time.perf_counter()
        if raw:
            if dev_inputs:
                rc = r_step_dev(hnd, img_ptr[i], Wpx, imu_ptr[i], imu_n[i], None, -1, 0, pose_ptr, valid_ptr)
            else:
                if prefetch and i + 1 < n_frames:
                    # the host announces frame i+1 when it arrives (System::PushImageData), i.e. while frame i is processed: its H2D
                    # copy runs on the library's copy stream inside THIS step's timed region (fenced before the end event below)
                    r_pref(hnd, img_ptr[i + 1], Wpx, Hpx, Wpx, 1)
                rc = r_step(hnd, img_ptr[i], Wpx, Hpx, Wpx, 1, imu_ptr[i], imu_n[i], None, -1, 0, pose_ptr, valid_ptr)
            if rc < 0:
                capi.check(rc, "rvio_vio_step")
            pose = pose_buf if valid.value else None
        elif dev_inputs:
            dc = (d_c2 if got_pose else d_c1)[i]
            pose = vio.step_dev(d_frames[i].data_ptr(), frames[i].shape[1], imus[i],
                                dc.data_ptr() if dc is not None else None, 0 if dc is None else dc.shape[0])
        else:
            if prefetch and i + 1 < n_frames:
                # the host announces frame i+1 when it arrives (System::PushImageData), i.e. while frame i is processed: its H2D
                # copy runs on the library's copy stream inside THIS step's timed region (fenced before the end event below)
                vio.prefetch(frames[i + 1])
            pose = vio.step(frames[i], imus[i], cands[i], device_detector=inloop)
        if timing:
            wall += time.perf_counter() - t0
            if prefetch:
                if raw:
                    r_fence(hnd, None)
                else:
                    vio.prefetch_fence()
            ev1[timed].record(stream)
            timed += 1
            L.rvio_vio_timeline(vio.h, 1 if stage_diag else 0, host_tl.ctypes.data)   # host wall clock of the step just finished: [6] enqueue, [7] blocked in the sync
            host_us.append((1e3 * float(host_tl[6]), 1e3 * float(host_tl[7])))
            if stage_diag:
                stages.append([1e3 * float(x) for x in host_tl[:6]])
            ui = vio.update_info()
            infos.append((int(ui.n_feat), int(ui.n_good), int(ui.rows_stacked), int(ui.rank), int(ui.rank_flags)))
        elif got_pose:
            warm += 1
        if pose is not None:
            got_pose = True
        i += 1
    torch.cuda.synchronize()
    _LAST_POSE["pose"] = None if pose is None else np.array(pose, np.float64)     # what the last timed step returned (--dump-outputs)
    step_ms = [a.elapsed_time(b) for a, b in zip(ev0, ev1)]
    # where a step's wall time goes on the host: inside the C call, enqueueing (image copy + graph launch) and blocked in its one
    # synchronisation; what is left of the wall time per step is the Python / ctypes layer around the call
    _LAST_DRIVE.update(host_enqueue_us=round(float(np.median([h[0] for h in host_us])), 1),
                       host_blocked_in_sync_us=round(float(np.median([h[1] for h in host_us])), 1),
                       wall_us=round(1e6 * wall / max(1, K), 1))
    if stage_diag:
        _LAST_DRIVE["stage_us"] = [round(float(v), 1) for v in np.median(np.array(stages), 0)]
    return step_ms, wall, L.rvio_b200_kernel_launches() - launches0, i, infos


def dump_outputs(directory, vio, pose, info):
    """--dump-outputs: what a caller of the device-resident path holds after the last timed step -- the pose it returned (NaN while
    the filter initialises), the filter state x / P read back from the handle, and the step's update counters (n_feat, accepted,
    stacked rows, rows kept, rank flags).  A few hundred kB at most (configs[4]: P is 204 x 204)."""
    x, P = vio.state()
    os.makedirs(directory, exist_ok=True)
    out = {"pose": np.full(7, np.nan) if pose is None else pose, "state_x": x, "state_P": P, "update_info": np.array(info)}
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, np.float64))


def run_b200(args, cfg, wl, rank, world, local_rank):
    import torch
    import ctypes as C
    from rvio_b200 import capi, host
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = bind_to_gpu_numa_node(local_rank)
    L = capi.lib()
    K, W = args.steps, args.warmup
    frames, imus = wl["frames"], wl["imus"]
    n_frames = len(frames)
    flush = torch.empty(384 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    inloop = args.detector == "inloop"

    import torch.distributed as dist
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- settling passes (untimed for the result, but timed and reported): the first few hundred frames a process pushes through the
    #      pipeline run slower than the same frames later (observed: the leg that happened to run first was ~50 us / step slower
    #      whatever its input mode), so the measured legs start from a settled process.  Alternating host-input / device-input passes
    #      of the same K-step protocol until at least RVIO_BENCH_SETTLE_STEPS (400) steps have run.
    settle = []
    want = int(os.environ.get("RVIO_BENCH_SETTLE_STEPS", "400"))
    done = 0
    while done < want and len(settle) < 24:
        mode_dev = len(settle) % 2 == 1
        vio = host.Vio(cfg, local_rank)
        ms, _, _, _, _ = drive(L, vio, wl, K, W, dev, inloop, mode_dev, flush)
        vio.close()
        settle.append(("device" if mode_dev else "host", round(float(np.mean(ms)), 4)))
        done += K + W
    with ClockSampler(local_rank) as clk:
        # ---- e2e legs (host buffers in pinned memory through the public C ABI).  `e2e`: the host announces frame k+1 while frame
        #      k is processed (rvio_vio_prefetch: the reference's System::PushImageData moment), so its upload overlaps frame k
        #      (headline `e2e`); `e2e.strict`: no announcement, every step uploads its own frame before it can start.
        vio = host.Vio(cfg, local_rank)
        barrier()
        e2s_ms, e2s_wall, _, _, _ = drive(L, vio, wl, K, W, dev, inloop, False, flush)
        host_e2s = dict(_LAST_DRIVE)
        barrier()
        vio.close()
        vio = host.Vio(cfg, local_rank)
        barrier()
        e2e_ms, e2e_wall, _, _, _ = drive(L, vio, wl, K, W, dev, inloop, False, flush, prefetch=True)
        host_e2e = dict(_LAST_DRIVE)
        pref_hits = vio.prefetch_fence()
        barrier()
        vio.close()
        # ---- device-resident leg (headline `value`)
        vio = host.Vio(cfg, local_rank)
        barrier()
        dev_ms, dev_wall, launches, used, infos = drive(L, vio, wl, K, W, dev, inloop, True, flush)
        host_dev = dict(_LAST_DRIVE)
        barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, vio, _LAST_POSE["pose"], infos[-1])
    # ---- bare H2D copy of one frame from pinned memory (what `e2e.sync` adds in front of every step)
    pin = torch.from_numpy(frames[0]).pin_memory(); dst = torch.empty(pin.shape, dtype=pin.dtype, device=dev)
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        dst.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    h0.record()
    for _ in range(20):
        dst.copy_(pin, non_blocking=True)
    h1.record(); torch.cuda.synchronize()
    h2d_frame_us = 1e3 * h0.elapsed_time(h1) / 20
    del pin, dst

    # ---- the headline numbers are complete here: reduce them over the ranks NOW, so that nothing an extra leg does can lose them
    t_dev = float(np.sum(dev_ms)) / 1e3
    t_e2e = float(np.sum(e2e_ms)) / 1e3
    t_e2s = float(np.sum(e2s_ms)) / 1e3
    t_dev_rank, t_e2e_rank = [t_dev], [t_e2e]
    if world > 1:
        t = torch.tensor([t_dev, t_e2e, t_e2s], dtype=torch.float64, device=dev)
        every = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(every, t)                                           # per-rank times: the slow rank is named in the JSON line
        t_dev_rank = [float(e[0]) for e in every]; t_e2e_rank = [float(e[1]) for e in every]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev, t_e2e, t_e2s = float(t[0]), float(t[1]), float(t[2])
    res = dict(t_dev=t_dev, t_e2e=t_e2e, t_e2s=t_e2s, dev_ms=dev_ms, e2e_ms=e2e_ms, launches=int(launches), clocks=clk.summary(),
               prof={}, dev_wall=dev_wall, e2e_wall=e2e_wall, e2s_wall=e2s_wall, timeline=None, batch=None, infos=infos,
               affinity=affinity, sharded=None, t_dev_rank=t_dev_rank, t_e2e_rank=t_e2e_rank, pref_hits=int(pref_hits),
               h2d_frame_us=h2d_frame_us, settle=settle, host_us={"value": host_dev, "e2e": host_e2e, "e2e.strict": host_e2s})
    _arm_legs_deadline(res, rank)

    # ---- per-stage timeline of the main stream (CUDA events inside the library), a few steps
    if rank == 0:
        tl = np.zeros(8, np.float32)
        L.rvio_vio_timeline(vio.h, 1, None)
        acc = []
        for i in range(used, min(used + 24, n_frames)):
            vio.step(frames[i], imus[i], wl["cand2"][i], device_detector=inloop)
            L.rvio_vio_timeline(vio.h, 1, tl.ctypes.data)
            acc.append(tl.copy())
        L.rvio_vio_timeline(vio.h, 0, None)
        used = min(used + 24, n_frames)
        res["timeline"] = dict(zip(["tracker", "feature+normal_terms", "wait_propagate", "solve", "augment_compose", "tail",
                                    "host_enqueue", "host_blocked_in_sync"],
                                   [round(float(v) * 1e3, 1) for v in np.median(np.array(acc), 0)]))
    # ---- per-kernel events over a few more steps (roofline leg)
    if rank == 0:
        prof = {}
        L.rvio_b200_profile(1)
        n_prof = 0
        for i in range(used, min(used + 24, n_frames)):
            vio.step(frames[i], imus[i], wl["cand2"][i], device_detector=inloop)
            n_prof += 1
        L.rvio_b200_profile(0)
        buf = C.create_string_buffer(1 << 16)
        nbytes = L.rvio_b200_profile_report(buf, len(buf))
        for line in buf.raw[:nbytes].decode().splitlines():
            name, cnt, tot = line.split()
            prof[name] = (int(cnt), float(tot), n_prof)
        res["prof"] = prof
    vio.close()
    barrier()
    # ---- batch leg (BASELINE configs[3]: independent streams, several per GPU, no communication): S handles driven by
    #      S host threads on the same device-resident frames; aggregate frames/s over the slowest stream (wall clock
    #      between device synchronisations; the single-stream `value` above is the CUDA-event number).
    S = args.batch_streams
    batch = None
    if S > 1:
        d_frames = [torch.from_numpy(f).to(dev) for f in frames]
        d_c1 = [torch.from_numpy(c).to(dev) if len(c) else None for c in wl["cand1"]]
        d_c2 = [torch.from_numpy(c).to(dev) if len(c) else None for c in wl["cand2"]]

    def run_batch():
        # Round 1 saw this leg stall under torchrun: eight host threads were CAPTURING frame graphs concurrently while an NCCL
        # process group (its watchdog / proxy threads) was alive.  Pre-roll and warm-up (which is where every frame graph of a
        # stream is captured) now run one stream after the other on the main thread; the worker threads only replay.
        vios = [host.Vio(cfg, local_rank) for _ in range(S)]
        Kb = min(K, 100)

        def one(v, i, got):
            dc = (d_c2 if got else d_c1)[i]
            if inloop:
                return v.step_dev(d_frames[i].data_ptr(), frames[i].shape[1], imus[i], None, -1)
            return v.step_dev(d_frames[i].data_ptr(), frames[i].shape[1], imus[i], dc.data_ptr() if dc is not None else None,
                              0 if dc is None else dc.shape[0])

        starts = []
        for v in vios:                                        # sequential pre-roll + warm-up (+ 4 steady frames: both graph parities exist)
            got, i, warm = False, 0, 0
            while not (got and warm >= W + 4):
                pose = one(v, i, got)
                if got:
                    warm += 1
                if pose is not None:
                    got = True
                i += 1
            starts.append(i)
        barrier()                                             # all ranks replay their streams at the same time
        start_bar = threading.Barrier(S + 1); end_bar = threading.Barrier(S + 1)
        errs = []

        def worker(v, i0):
            try:
                start_bar.wait(timeout=240)
                for k in range(Kb):
                    one(v, i0 + k, True)
                end_bar.wait(timeout=240)
            except Exception as e:          # pragma: no cover
                errs.append(e)
                try:
                    start_bar.abort(); end_bar.abort()
                except Exception:
                    pass

        if max(starts) + Kb > n_frames:
            errs.append(RuntimeError("stream too short for the batch leg"))
        ths = [threading.Thread(target=worker, args=(v, i0)) for v, i0 in zip(vios, starts)]
        t0 = t1 = 0.0
        if not errs:
            for t in ths:
                t.start()
            try:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                start_bar.wait(timeout=240)
                end_bar.wait(timeout=240)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
            except threading.BrokenBarrierError:                  # a worker failed (or timed out): no batch number, no hang
                errs.append(RuntimeError("batch leg aborted"))
            for t in ths:
                t.join(timeout=60)
        for v in vios:
            v.close()
        if errs:
            return None
        return S * Kb / (t1 - t0), Kb

    # Programmatic dependent launch keeps the NEXT kernel of a stream resident (and its shared memory / registers taken) while the
    # current one runs: a gain for one stream that leaves most of the GPU idle, a cost when eight streams compete for the SMs.  The leg
    # is therefore run in both settings (rvio_b200_pdl is a process-wide switch a multi-stream host would set) and reports both.
    if S > 1:
        pdl0 = L.rvio_b200_pdl(-1)
        both = {}
        for setting in (pdl0, 1 - pdl0):
            L.rvio_b200_pdl(setting)
            try:
                r = run_batch()
            except Exception:          # pragma: no cover
                r = None
            both["on" if setting else "off"] = r
        L.rvio_b200_pdl(pdl0)
        vals = {k: (v[0] if v else 0.0) for k, v in both.items()}
        oks = {k: (1.0 if v else 0.0) for k, v in both.items()}
        if world > 1:
            # every rank takes part in the same collectives, whatever happened to its own batch leg (a rank that skipped one
            # would leave the others waiting in NCCL for ever)
            bt = torch.tensor([vals["on"], vals["off"], oks["on"], oks["off"]], dtype=torch.float64, device=dev)
            dist.all_reduce(bt, op=dist.ReduceOp.SUM)
            vals = {"on": float(bt[0]), "off": float(bt[1])}
            oks = {"on": float(bt[2]) / world, "off": float(bt[3]) / world}
        good = {k: v for k, v in vals.items() if oks[k] == 1.0}
        if good:
            best = max(good, key=good.get)
            Kb = next(v[1] for v in both.values() if v) if any(both.values()) else min(K, 100)
            batch = {"streams_per_gpu": S, "steps_per_stream": Kb, "value": good[best], "unit": "frames/s", "n_gpus": world, "pdl": best,
                     "by_pdl_setting": {k: round(v, 1) for k, v in good.items()},
                     "timing": "wall clock between device synchronisations, all streams concurrent (graphs captured beforehand, one stream at a time)"}
    res["batch"] = batch
    # ---- feature-sharded single stream (BASELINE configs[4]: 2048 features, 30-clone window): every rank is fed the same
    #      frames; LK all-gather + normal-term all-reduce are enqueued by the library on its own stream (in the frame graph)
    if world > 1 and not args.no_sharded:
        try:
            res["sharded"] = sharded_leg(args, L, dev, flush, rank, world, local_rank)
        except Exception as e:          # pragma: no cover
            res["sharded"] = {"error": repr(e)[:300]}
        barrier()
    return res


def update_cost_model(rows_per_feat, n, d):
    """SURVEY 8(d) accounting for one Updater::update: fp32-equivalent flops (Householder accounting for the compression)
    and algorithmic bytes (float64 here: H written once, read by the gate and by the compression; P in + out)."""
    r = np.asarray(rows_per_feat, np.float64)
    R = float(r.sum())
    f_gate = float((2 * r * n * n + 2 * r * r * n).sum())
    f_qr = max(0.0, 2 * R * n * n - (2.0 / 3.0) * n ** 3) if R > n else 0.0
    rk = min(R, n)
    f_ekf = 4 * d ** 3 + 2 * d * d * rk + 2 * rk ** 3 + 4 * d * n * rk + 2 * d * rk * rk + 2 * rk * n * n + 2 * rk * rk * n
    return dict(R=int(R), flops=f_gate + f_qr + f_ekf, f_gate=f_gate, f_qr=f_qr, f_ekf=f_ekf,
                bytes=8.0 * R * n * 3 + 16.0 * d * d)


UPDATE_KERNELS = ("k_feature", "k_gate", "k_gram", "k_rank_rule", "k_givens_ref", "k_wgemm", "k_gj_block", "k_pout_finalize", "k_dgemm",
                  "k_gauss_jordan", "k_finalize", "k_chol", "k_tsqr")


def _profile_report(L):
    import ctypes as C
    buf = C.create_string_buffer(1 << 16)
    nbytes = L.rvio_b200_profile_report(buf, len(buf))
    out = {}
    for line in buf.raw[:nbytes].decode().splitlines():
        name, cnt, tot = line.split()
        out[name] = (int(cnt), float(tot))
    return out


def update_worstcase_leg(L, dev, flush, peaks, idx, reps=4):
    """SURVEY 8(d) updater micro-benchmark: F_u maximum-length type-'1' tracks (the tallest stacked H of the config):
    14 700 x 150 (configs[2]) and 60 416 x 180 (configs[4]).  Per-kernel CUDA events inside the library; the update-kernel
    roofline is algorithmic bytes / flops of the whole update over the summed kernel time."""
    import torch
    from rvio_b200 import synth, host
    cfg = synth.baseline_config(idx)
    Fu = (cfg.n_features + 1) // 2
    x, P, types, off, xy = synth.make_update_case(cfg, Fu, 900 + idx, mix_types=False)
    N = cfg.max_track_len - 1; n = 6 * N; d = 24 + n
    upd = host.Updater(cfg, dev.index)
    for _ in range(2):
        upd.update(x, P, types, (off, xy))
    info = upd.info
    dof = upd.debug(len(types))["dof"]
    L.rvio_b200_profile(1)
    wall = []
    for r in range(reps):
        flush.fill_(r); torch.cuda.synchronize()
        t0 = time.perf_counter()
        upd.update(x, P, types, (off, xy))
        wall.append(time.perf_counter() - t0)
    L.rvio_b200_profile(0)
    prof = _profile_report(L)
    upd.close()
    per = {k: v[1] / reps for k, v in prof.items()}                        # ms per update
    t_upd = sum(v for k, v in per.items() if any(k.startswith(u) for u in UPDATE_KERNELS)) / 1e3
    cm = update_cost_model(dof[dof > 0], n, d)
    gbs = cm["bytes"] / t_upd / 1e9
    tfl = cm["flops"] / t_upd / 1e12
    top = max(per, key=per.get)
    return {"workload": f"BASELINE configs[{idx}] worst-case update: {Fu} type-'1' tracks of length {cfg.max_track_len}, N={N} clones, "
                        f"stacked H {cm['R']} x {n}, float64", "n_good": int(info.n_good), "rows": int(info.rows_stacked),
            "rank": int(info.rank), "rank_flags": int(info.rank_flags),
            "ms_update_kernels": 1e3 * t_upd, "ms_through_c_abi": 1e3 * float(np.median(wall)),
            "updates_per_s": 1.0 / t_upd,
            "roofline_update": {"bound": "hbm", "algorithmic_bytes": cm["bytes"], "flops": cm["flops"],
                                "flops_split": {"gate": cm["f_gate"], "compression_householder": cm["f_qr"], "ekf": cm["f_ekf"]},
                                "achieved": gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                                "tflops": tfl, "tensor_peak_tflops_bf16": peaks.get("bf16_tflops"),
                                "frac_of_tensor_peak": tfl / peaks["bf16_tflops"] if peaks.get("bf16_tflops") else None,
                                "top_kernel": top},
            "kernel_us_per_update": {k: round(v * 1e3, 1) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}}


def sharded_leg(args, L, dev, flush, rank, world, local_rank):
    """BASELINE configs[4]: ONE stream, 2048 features / 30 clones, feature-sharded over the N GPUs (SURVEY 8e).  Value =
    frames/s of that stream (max over ranks of the device time); rank 0 afterwards runs the same stream unsharded."""
    import torch
    import torch.distributed as dist
    import rvio_b200  # noqa: F401
    from rvio_b200 import synth, host
    cfg = synth.baseline_config(4)
    Ks, Ws = min(args.steps, 20), cfg.max_track_len + 6
    wl = make_workload(cfg, int(T_STATIC * cfg.fps) + 4 + Ws + Ks + 20, SHARDED_SEED, False)  # same seed on every rank: same frames
    uid = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        uid.copy_(torch.frombuffer(bytearray(host.nccl_unique_id()), dtype=torch.uint8))
    dist.broadcast(uid, 0)
    vio = host.Vio(cfg, local_rank)
    vio.shard_init(rank, world, bytes(uid.cpu().numpy().tobytes()))
    ag_us, ar_us = vio.shard_probe(50)
    dist.barrier(); torch.cuda.synchronize()
    ms, _, launches, used, infos = drive(L, vio, wl, Ks, Ws, dev, True, True, flush)
    glaunch = vio.graph_launches()
    vio.close()
    t = torch.tensor([float(np.sum(ms)) / 1e3], dtype=torch.float64, device=dev)
    every = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(every, t)
    tmax = max(float(e[0]) for e in every)
    out = {"workload": f"BASELINE configs[4]: one synthetic {cfg.width}x{cfg.height} stream, {cfg.n_features} features, {cfg.max_track_len - 1}-clone window, "
                       f"feature-sharded over {world} GPUs (LK all-gather + normal-term all-reduce in stream)",
           "n_gpus": world, "steps": Ks, "warmup": Ws, "value": Ks / tmax, "unit": "frames/s", "ms_per_step": 1e3 * tmax / Ks,
           "per_rank_ms_per_step": [round(1e3 * float(e[0]) / Ks, 4) for e in every],
           "collectives_us_per_frame": {"allgather_lk": round(ag_us, 2), "allreduce_normal_terms": round(ar_us, 2),
                                        "bytes": {"allgather": 17 * ((cfg.n_features + world - 1) // world) * world,
                                                  "allreduce": 8 * ((6 * (cfg.max_track_len - 1)) ** 2 + 2 * 6 * (cfg.max_track_len - 1) + 9)}},
           "graph_replays": glaunch, "gpu_launches": int(launches),
           "update_frames": [list(x) for x in infos[:8]]}
    out["undecided_rank_rule_frames"] = int(sum(1 for x in infos if x[4] & 4))
    if rank == 0:
        # The same stream on ONE GPU, twice.  (a) In the reference rule, as the sharded form runs: where the rank-rule certificate cannot
        # decide, the single-GPU path replays the reference's Givens sweep over the stacked rows (k_givens_ref: ~10^3 dependent steps),
        # which the sharded form cannot do -- its rows are distributed -- so it keeps every row and says so (RVIO_RANK_UNDECIDED; same
        # x+ / P+ whenever the reference's cut would not have discarded anything, which tests/dist_sharded_vio.py checks on this stream).
        # (b) With every row kept on every frame (RVIO_RANK_RULE_FULL_INFORMATION): the same arithmetic per frame as the sharded run, so
        # THIS ratio is what the sharding itself buys; (a) additionally contains the cost of the sweep.
        for key, full, ratio in (("unsharded_same_stream", False, "speedup_vs_1gpu"),
                                 ("unsharded_all_rows_kept", True, "speedup_vs_1gpu_same_rows_kept")):
            try:                                           # a failure here must not cost the sharded numbers above
                ref = host.Vio(cfg, local_rank)
                if full:
                    ref.set_rank_rule(True)
                ms1, _, _, _, inf1 = drive(L, ref, wl, Ks, Ws, dev, True, True, flush)
                ref.close()
                out[key] = {"value": Ks / (float(np.sum(ms1)) / 1e3), "ms_per_step": float(np.mean(ms1)),
                            "undecided_rank_rule_frames": int(sum(1 for x in inf1 if x[4] & 4)),
                            "frames_resolved_by_givens_sweep": int(sum(1 for x in inf1 if x[4] & 2))}
                out[ratio] = (float(np.sum(ms1)) / 1e3) / tmax
            except Exception as e:                         # pragma: no cover
                out[key] = {"error": repr(e)[:200]}
    return out


def stress_leg(args, L, dev, flush, peaks, rank):
    """BASELINE configs[2]: 1280x720 frames, 600 features, 25-clone window on one GPU (short stream: the window must fill)."""
    import rvio_b200  # noqa: F401
    from rvio_b200 import synth, host
    cfg = synth.baseline_config(2)
    Ks, Ws = 10, cfg.max_track_len + 6
    wl = make_workload(cfg, int(T_STATIC * cfg.fps) + 4 + Ws + Ks + 20, SEED + 2, args.detector == "precomputed")
    inloop = args.detector == "inloop"
    vio = host.Vio(cfg, dev.index)
    e2e_ms, _, _, _, _ = drive(L, vio, wl, Ks, Ws, dev, inloop, False, flush)
    vio.close()
    vio = host.Vio(cfg, dev.index)
    dev_ms, _, launches, used, infos = drive(L, vio, wl, Ks, Ws, dev, inloop, True, flush)
    L.rvio_b200_profile(1)
    n_prof = 0
    for i in range(used, min(used + 4, len(wl["frames"]))):
        vio.step(wl["frames"][i], wl["imus"][i], wl["cand2"][i], device_detector=inloop)
        n_prof += 1
    L.rvio_b200_profile(0)
    prof = _profile_report(L)
    vio.close()
    per = {k: v[1] / max(n_prof, 1) for k, v in prof.items()}
    N = cfg.max_track_len - 1; n = 6 * N; d = 24 + n
    return {"workload": f"BASELINE configs[2]: synthetic {cfg.width}x{cfg.height} stream, {cfg.n_features} features, {N}-clone window",
            "steps": Ks, "warmup": Ws, "value": Ks / (float(np.sum(dev_ms)) / 1e3), "unit": "frames/s",
            "ms_per_step": float(np.mean(dev_ms)), "e2e": {"value": Ks / (float(np.sum(e2e_ms)) / 1e3), "unit": "frames/s",
                                                            "h2d_bytes_per_step": cfg.width * cfg.height + 10 * 64},
            "gpu_launches": int(launches), "update_frames": [list(t) for t in infos],
            "kernel_us_per_step": {k: round(v * 1e3, 1) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}}


def roofline_from_profile(prof, cfg, peaks):
    if not prof:
        return None, {}
    per_step = {k: v[1] / v[2] for k, v in prof.items()}                   # ms per step per kernel
    total = sum(per_step.values())
    # the dominant kernel of the frame's CRITICAL PATH: the side-stream kernels (propagation, the detector chain, FindNewer) run
    # beside it and end before it (DESIGN.md section 7)
    off_path = ("k_propagate", "k_det_eig", "k_det_nms", "k_det_select", "k_det_subpix", "k_find_newer_refill")
    on_path = {k: v for k, v in per_step.items() if k not in off_path} or per_step
    top = max(on_path, key=on_path.get)
    cnt, tot_ms, n_steps = prof[top]
    avg_s = tot_ms / cnt / 1e3
    W, H, F = cfg.width, cfg.height, cfg.n_features
    N = cfg.max_track_len - 1
    n, d = 6 * N, 24 + 6 * N
    # algorithmic bytes per launch (DESIGN.md "Kernels"): what the kernel must move at least once
    alg = {
        "k_lk": 2 * 1.328 * W * H + 20 * F,                                 # both pyramids read once + per-feature I/O
        "k_clahe_apply": W * H + 1.0 * W * H,                               # read raw, write level 0
        "k_clahe_lut": W * H,
        "k_pyr_down": 1.25 * W * H,                                         # all three launches together ~ read+write 0.33WH
        "k_pyr_down3": 1.33 * W * H,                                        # level 0 read once, levels 1-3 written
        "k_update_small": 8.0 * (n * n + 3 * d * d),                        # G in, P in, P out (+ the copy of P the epilogue reads)
        "k_ransac_bookkeep": 40.0 * F,
        "k_feature": 8.0 * (n * n) + 8.0 * ((F + 1) // 2) * 2 * (N + 1) * n,  # Pcc once + projected blocks written
        "k_gram": 8.0 * ((F + 1) // 2) * 2 * (N + 1) * n,
        "k_gauss_jordan": 8.0 * (n * n + n * (d + 1)) * 2,
        "k_dgemm": 8.0 * 3 * d * d,
        "k_propagate": 8.0 * 2 * d * d,
        "k_det_eig": 5.0 * W * H,                                         # equalised frame read once, float map written
        "k_det_nms": 4.0 * W * H,
        "k_det_select": 2 * 8.0 * 0.053 * W * H,                          # candidate keys (5.3% of the pixels are local maxima on this stream), read twice
        "k_det_subpix": F * 30 * 18.0 * 18.0,                             # source window per corner and iteration
        "k_augment_compose": 8.0 * 2 * d * d,
    }.get(top, None)
    rf = {"kernel": top, "bound": "hbm", "launches_per_step": cnt / n_steps, "avg_launch_us": avg_s * 1e6,
          "share_of_step_kernel_time": per_step[top] / total if total else None,
          "peak": peaks.get("hbm_gbs"), "unit": "GB/s", "traffic": None,
          "peak_source": "MEASURED_PEAKS.json (measured)" if peaks.get("_measured") else "fallback 6650 GB/s"}
    if alg is not None:
        rf["algorithmic_bytes_per_launch"] = alg
        rf["achieved"] = alg / avg_s / 1e9
        rf["frac"] = rf["achieved"] / rf["peak"] if rf["peak"] else None
    try:                                                                    # measured DRAM traffic of the same kernel (committed ncu summary)
        import glob
        tr = json.load(open(sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic_r*.json")))[-1]))
        rf["traffic"] = tr["bytes_per_launch"].get(top)
        rf["traffic_source"] = tr["source"]
    except Exception:
        pass
    rf["note"] = ("single-stream VIO at this size moves ~2 MB and ~50 MFLOP per frame: every kernel is latency-bound, "
                  "the roofline fraction is reported for completeness (SURVEY 8d)")
    return rf, {k: round(v * 1e3, 2) for k, v in sorted(per_step.items(), key=lambda kv: -kv[1])}   # us per step


# ----------------------------------------------------------------------------------------- reference arm
def run_reference(cfg, wl, steps, warmup, threads, inloop=True):
    """Same frame loop on the host: cv2 (real OpenCV) for CLAHE / pyramidal LK, oracle C port for the Eigen stages."""
    import ctypes as C
    import cv2
    from oracle import oracle as orc
    cv2.setNumThreads(threads)
    L = orc.lib()
    v = orc.VioOracle(cfg)
    trk = v.tracker
    clahe = cv2.createCLAHE(3.0, (5, 5))
    crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 1e-2)
    H, Wd = cfg.height, cfg.width
    frames, imus = wl["frames"], wl["imus"]
    state = dict(last_eq=None)

    def track(img, imu, cand1, cand2):
        # Tracker::track with the OpenCV stages through cv2 (Tracker.cc:198-202,237-244)
        eq = cv2.createCLAHE(3.0, (5, 5)).apply(img) if cfg.enable_equalizer else img     # new object per frame, as the reference
        n = L.orc_tracker_n_feats(trk.h)
        if state["last_eq"] is not None and n > 0:
            pts = np.ctypeslib.as_array(L.orc_tracker_feats(trk.h), (n, 2)).copy()
            nxt, stt, _ = cv2.calcOpticalFlowPyrLK(state["last_eq"], eq, pts, None, winSize=(15, 15), maxLevel=3, criteria=crit,
                                                   flags=0, minEigThreshold=1e-3)
            lk = np.ascontiguousarray(nxt.reshape(-1, 2), np.float32); stt = np.ascontiguousarray(stt.reshape(-1), np.uint8)
        else:
            lk = np.zeros((1, 2), np.float32); stt = np.zeros(1, np.uint8)
        rc = L.orc_tracker_track_ext(trk.h, np.ascontiguousarray(eq), lk, stt, np.ascontiguousarray(imu), len(imu))
        if rc == 2:
            return
        if inloop:                                                     # FeatureDetector::DetectWithSubPix through cv2, as the reference calls it
            if rc == 1:
                cand1 = orc.detect_with_subpix(eq, cfg.n_features, 1, cfg)             # Tracker.cc:207
            elif L.orc_tracker_n_free(trk.h) > 0:
                cand2 = orc.detect_with_subpix(eq, cfg.n_features, 2, cfg)             # Tracker.cc:350
        if rc == 1:
            if len(cand1):
                L.orc_tracker_seed(trk.h, np.ascontiguousarray(cand1, np.float32), len(cand1))
        elif L.orc_tracker_n_free(trk.h) > 0 and len(cand2):
            nt = L.orc_tracker_n_tracked(trk.h)
            ref = np.ctypeslib.as_array(L.orc_tracker_tracked_px(trk.h), (max(nt, 1), 2))[:nt].copy()
            newer = orc.find_newer(cfg, cand2, ref)
            if len(newer):
                L.orc_tracker_refill(trk.h, newer, len(newer))
        L.orc_tracker_commit(trk.h)
        state["last_eq"] = eq

    trk.track = lambda img, imu: None      # VioOracle.step calls tracker.track(img, imu): replaced per frame below
    got_pose, warm, timed, i = False, 0, 0, 0
    t_total = 0.0
    per = []
    while timed < steps and i < len(frames):
        c1, c2 = wl["cand1"][i], wl["cand2"][i]
        trk.track = (lambda img, imu, c1=c1, c2=c2: track(img, imu, c1, c2))
        timing = got_pose and warm >= warmup
        t0 = time.perf_counter()
        pose = v.step(frames[i], imus[i])
        dt = time.perf_counter() - t0
        if timing:
            t_total += dt; per.append(dt); timed += 1
        elif got_pose:
            warm += 1
        if pose is not None:
            got_pose = True
        i += 1
    tm = np.array(v.timing[-timed:]) if timed else np.zeros((0, 2))
    return dict(t=t_total, steps=timed, tracker_ms=float(np.median(tm[:, 0])) if timed else None,
                filter_ms=float(np.median(tm[:, 1])) if timed else None)


# ----------------------------------------------------------------------------------------- main
def _watchdog(seconds):
    """A wedged run (driver, NCCL, a kernel that never returns) must not hold the GPU box until the caller's limit: dump
    every thread's stack and exit non-zero after `seconds`."""
    import faulthandler
    faulthandler.dump_traceback_later(seconds, exit=True)


# The headline numbers (value, e2e) are complete before any extra leg (timeline, per-kernel profile, batch, sharded stream,
# stress stream, worst-case updates, CPU baseline) starts.  Should one of those legs wedge (a collective that never returns on
# some box), the JSON line is still printed from what exists, with the unfinished legs named, and every rank exits 0.
_LINE_CTX = {}
_DEADLINE = {"timer": None, "res": None}


def _arm_legs_deadline(res, rank):
    seconds = float(os.environ.get("RVIO_BENCH_LEGS_DEADLINE_S", "420"))
    _DEADLINE["res"] = res

    def fire():                                               # pragma: no cover
        import faulthandler
        faulthandler.dump_traceback(file=sys.stderr)
        if rank == 0:
            try:
                out = build_line(_DEADLINE["res"])
                out["legs_deadline"] = f"extra legs did not finish within {seconds:.0f} s: line printed from the completed legs"
                print(json.dumps(out), flush=True)
            finally:
                os._exit(0)
        time.sleep(3.0)
        os._exit(0)

    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    _DEADLINE["timer"] = t


def _disarm_legs_deadline():
    if _DEADLINE["timer"] is not None:
        _DEADLINE["timer"].cancel()
        _DEADLINE["timer"] = None


def build_line(res):
    """The JSON line from whatever legs have completed (`res` is filled leg by leg)."""
    c = _LINE_CTX
    cfg, wl, world, K, W, peaks = c["cfg"], c["wl"], c["world"], c["K"], c["W"], c["peaks"]
    rf, per_kernel_us = roofline_from_profile(res["prof"], cfg, peaks)
    n_imu = int(np.median([len(x) for x in wl["imus"][-K:]]))
    n_cand = int(np.median([len(x) for x in wl["cand2"][-K:]]))
    h2d = cfg.width * cfg.height + n_imu * 64 + n_cand * 8
    d2h = 56 + 4 * 46 + 64
    value = world * K / res["t_dev"]
    e2e = world * K / res["t_e2e"]                            # headline e2e: frames announced one step ahead (upload inside the timed region)
    out = {"metric": "vio_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": 1e3 * res["t_dev"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic", "config": c["workload"],
           "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "ms_per_step": 1e3 * res["t_e2e"] / K, "wall_ms_per_step": 1e3 * res["e2e_wall"] / K,
                   "upload": "host frames in pinned memory through the C ABI.  Frame k+1 is announced at the start of step k "
                             "(rvio_vio_prefetch = the moment the reference's host queues it, System::PushImageData): its H2D copy runs on "
                             "the library's copy stream beside frame k, INSIDE step k's timed region (the end event is recorded after "
                             "rvio_vio_prefetch_fence); so every timed step contains exactly one frame upload, the IMU rows going up and the "
                             "pose / counters coming back",
                   "steps_fed_by_prefetch": res["pref_hits"],
                   "strict": {"value": world * K / res["t_e2s"], "unit": "frames/s", "ms_per_step": 1e3 * res["t_e2s"] / K,
                              "wall_ms_per_step": 1e3 * res["e2s_wall"] / K,
                              "what": "no announcement: every step uploads ITS OWN frame (pinned, DMA straight into the gray buffer) before its "
                                      "first kernel can start -- one isolated H2D transfer costs ~50 us of latency on these boxes"},
                   "h2d_frame_us": round(res["h2d_frame_us"], 2)},
           "gpu_launches": res["launches"], "clocks": res["clocks"], "roofline": rf,
           "kernel_us_per_step": per_kernel_us, "stage_us_per_step": res["timeline"],
           "wall_ms_per_step": 1e3 * res["dev_wall"] / K, "batch": res["batch"], "sharded": res["sharded"]}
    out["parallelism"] = f"{world} independent stream(s), one per GPU (no collective on the data path)"
    out["per_rank_ms_per_step"] = {"device": [round(1e3 * t / K, 4) for t in res["t_dev_rank"]],
                                   "e2e": [round(1e3 * t / K, 4) for t in res["t_e2e_rank"]]}
    out["cpu_affinity"] = res["affinity"]
    out["settle_passes_ms_per_step"] = res.get("settle")      # (input mode, mean ms / step) of the untimed passes before the measured legs
    out["host_us_per_step"] = res.get("host_us")              # per leg: C-call enqueue / blocked-in-sync / whole Python-level wall time
    try:
        from rvio_b200 import capi as _capi
        out["pdl"] = bool(_capi.lib().rvio_b200_pdl(-1))      # programmatic dependent launch between the frame's short dependent kernels
    except Exception:                                          # pragma: no cover
        out["pdl"] = None
    out["update_frames"] = {"rows_kept_flags": [list(t) for t in res["infos"][:32]],
                            "note": "(n_feat, accepted, stacked rows, rows kept by the reference's rank rule, flags) per timed step; the "
                                    "device runs the reference rule (RVIO_RANK_RULE_REFERENCE), the mode the parity tests cover"}
    for k in ("stress", "update_worstcase", "cpu_baseline"):
        if k in res:
            out[k] = res[k]
    return out


def main():
    args = parse()
    _watchdog(int(os.environ.get("RVIO_BENCH_WATCHDOG_S", "780")))
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import rvio_b200  # noqa: F401
    from rvio_b200 import synth
    cfg = synth.baseline_config(args.config)
    K, W = args.steps, max(args.warmup, 3)
    args.warmup = W
    n_frames = int(T_STATIC * cfg.fps) + 4 + W + K + 80        # pre-roll (first pose ~ frame 21), warm-up, timed steps, 2 x 24 steps of the timeline / profile legs
    workload = {"workload": f"BASELINE configs[{args.config}]: synthetic EuRoC-shaped {cfg.width}x{cfg.height} mono + 200 Hz IMU stream, "
                            f"{cfg.n_features} features, {cfg.max_track_len - 1}-clone window, 1 frame per step",
                "detector": ("FeatureDetector::DetectWithSubPix inside every timed step (whole Tracker::track): device kernels in this arm, "
                             "cv2.goodFeaturesToTrack + cornerSubPix in the reference arm; FindNewer + refill inside the step"
                             if args.detector == "inloop" else
                             "corner candidates pre-computed (cv2.goodFeaturesToTrack on the equalised frame), identical for both arms; "
                             "FindNewer + refill inside the timed step"),
                "l2": "384 MB device buffer rewritten between timed iterations (outside the per-step event pair)",
                "precision": "tracker bit-exact integer/float32, filter float64"}
    ncores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return
        wl = make_workload(cfg, int(T_STATIC * cfg.fps) + 4 + W + K + 30, SEED + args.config, args.detector == "precomputed")
        r = run_reference(cfg, wl, K, W, ncores, args.detector == "inloop")
        fps = r["steps"] / r["t"]
        out = {"metric": "vio_frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": r["steps"], "warmup": W,
               "ms_per_step": 1e3 * r["t"] / r["steps"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f64", "data": "synthetic", "impl": "reference", "config": workload,
               "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": ncores, "kind": "port",
                                "sample": f"{r['steps']} frames of the same stream; OpenCV stages via cv2 {__import__('cv2').__version__} "
                                          f"({ncores} threads), Eigen stages via oracle C port (1 thread, as the reference); "
                                          f"median tracker {r['tracker_ms']:.3f} ms, filter {r['filter_ms']:.3f} ms"},
               "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "gpu_launches": 0}
        print(json.dumps(out))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a B200: there is no CPU fallback")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = make_workload(cfg, n_frames, SEED + args.config + 1000 * rank + int(os.environ.get("RVIO_BENCH_SEED_OFFSET", "0")),
                       args.detector == "precomputed")
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peaks["_measured"] = True
    except Exception:
        peaks = {"hbm_gbs": 6650.0, "_measured": False}
    _LINE_CTX.update(cfg=cfg, wl=wl, world=world, K=K, W=W, peaks=peaks, workload=workload)
    res = run_b200(args, cfg, wl, rank, world, local_rank)
    if rank != 0:
        _disarm_legs_deadline()
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    if world == 1 and not args.no_extra_legs:
        import torch as _t
        from rvio_b200 import capi as _capi
        dev = _t.device("cuda", local_rank)
        fl = _t.empty(384 << 20, dtype=_t.uint8, device=dev)
        Lb = _capi.lib()
        try:
            res["stress"] = stress_leg(args, Lb, dev, fl, peaks, rank)
        except Exception as e:          # pragma: no cover
            res["stress"] = {"error": repr(e)[:200]}
        res["update_worstcase"] = {}
        for idx in (2, 4):
            try:
                res["update_worstcase"][f"configs[{idx}]"] = update_worstcase_leg(Lb, dev, fl, peaks, idx)
            except Exception as e:      # pragma: no cover
                res["update_worstcase"][f"configs[{idx}]"] = {"error": repr(e)[:200]}
        del fl
    if not args.no_cpu_baseline and world == 1:
        steps = 60
        wl2 = {k: (v[:int(T_STATIC * cfg.fps) + 4 + W + steps + 4] if isinstance(v, list) else v) for k, v in wl.items()}
        r = run_reference(cfg, wl2, steps, min(W, 10), ncores, args.detector == "inloop")
        import cv2
        res["cpu_baseline"] = {"value": r["steps"] / r["t"], "unit": "frames/s", "cores": ncores, "kind": "port",
                               "sample": f"{r['steps']} frames of the same stream; OpenCV stages via cv2 {cv2.__version__} ({ncores} threads), "
                                         f"Eigen stages via oracle C port (1 thread); median tracker {r['tracker_ms']:.3f} ms, filter {r['filter_ms']:.3f} ms"}
    _disarm_legs_deadline()
    print(json.dumps(build_line(res)), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
