#!/usr/bin/env python
"""bench.py -- headline benchmark of the grayskull hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c5|ops|match|tmatch] [--impl reference]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] ("c2"): gs_blur r=5 + gs_sobel on 4096x4096 synthetic
uint8 frames, batch 256 per GPU (weak scaling: every rank processes its own 256 frames; frames are
independent, no data-path collective).  A step = one pass of both ops over the batch.

One JSON line on stdout (rank 0):
  value      Mpixels/s, whole job, inputs resident in HBM, CUDA-event time, max over ranks
  e2e        the same metric through the C ABI with HOST (pinned) buffers: H2D + kernels + D2H in
             the timed region, chunked over two streams; e2e_dropin = the reference's own call shape
             (gs_blur / gs_sobel with plain host pointers, one image per call)
  roofline   dominant kernel's algorithmic HBM bytes / its own CUDA-event time vs MEASURED_PEAKS.json
  configs    BASELINE configs[2] (c3: gs_orb_extract, 1920x1080 x 1024) and configs[3] (c4: gs_integral +
             gs_lbp_detect, 3840x2160 x 256) measured in the same run: value, dominant kernel, roofline,
             clocks and their own cpu_baseline
  shard      BASELINE configs[4] (c5): one NCCL scatter of uint8 frames from rank 0 -> the frame pipeline on
             every rank -> one NCCL gather of the results; Mpixels/s including and excluding the collectives
  cpu_baseline  the reference's own C code (oracle/_ref, built from /root/reference) timed on this
             box's host cores on a bounded sample of the same workload
With --impl reference the whole line is the reference CPU arm (rank 0 only).

--steps K is the number of timed steps of the GPU arm.  The reference arm (--impl reference) runs at most K, as many
as fit its time budget, and reports the count it ran.

--dump-outputs DIR writes, right after the timed steps of the headline workload, what its last step computed
(the arrays a caller of that path receives) as DIR/<name>.npy: float32 for 8/16-bit data, float64 for 32-bit
words (exact), rows past a per-frame count zeroed.  DUMP_BYTES is shared out smallest output first, each taking all
of itself or an equal part of what is left; an output larger than its part is replaced by a fixed sample, the
sorted flat indices np.random.default_rng(0).integers(0, numel, k).  Inputs are seeded, so two builds run with the
same arguments can be compared array for array.  c3, c4 and tmatch blur their seeded noise with the build's own
gs_blur before timing, so a change to gs_blur also changes those workloads' inputs.  Rank 0 only.
"""
import argparse
import ctypes as C
import json
import math
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

W2, H2, B2, R2 = 4096, 4096, 256, 5            # c2
W3, H3, B3, NK3, T3 = 1920, 1080, 1024, 1250, 20   # c3
W4, H4, B4 = 3840, 2160, 256                  # c4 (sf 1.1, scales 1..4, step 2, max_rects 65536)
B5 = 1024                                     # c5: 8192 frames over 8 GPUs
NWIN4 = 30016520                              # windows per UHD frame (SURVEY.md 8d; checked against the library)
FALLBACK_HBM_GBS = 6650.0
DUMP_BYTES = 60_000_000                       # --dump-outputs: array data of all files together (headers stay under 64 MB)
NVLINK_GBS = 900.0                            # NVLink 5 per direction per GPU: the root's egress / ingress bound

METRICS = {
    "c2": ("Mpixels/s, gs_blur(r=5) + gs_sobel, 4096x4096 uint8", "Mpixels/s", 1e-6),
    "c3": ("Mpixels/s, gs_orb_extract (FAST-9 t=20 + BRIEF-256, nkps=1250), 1920x1080 uint8", "Mpixels/s", 1e-6),
    "c4": ("LBP cascade windows/s, gs_integral + gs_lbp_detect frontalface, 3840x2160", "windows/s", 1.0),
    "c5": ("Mpixels/s, pipeline blur(r=5) -> sobel -> gs_orb_extract -> gs_integral + gs_lbp_detect, 1920x1080 uint8", "Mpixels/s", 1e-6),
}


def workload_cfg(wl, n):
    """the `config` object of a workload -- shared by the GPU arm and the reference arm"""
    if wl == "c2":
        return {"workload": "c2: gs_blur r=5 + gs_sobel, 4096x4096 synthetic uint8, batch %d per GPU" % n,
                "frames_per_gpu": n, "l2": "inputs (%.1f GiB per GPU) exceed the 126 MB L2" % (n * H2 * W2 / 2**30)}
    if wl == "c3":
        return {"workload": "c3: gs_orb_extract nkps=1250 t=20, 1920x1080 blurred-noise uint8, batch %d per GPU" % n,
                "frames_per_gpu": n, "l2": "inputs (%.1f GiB per GPU) exceed the 126 MB L2" % (n * H3 * W3 / 2**30)}
    if wl == "c4":
        return {"workload": "c4: gs_integral + gs_lbp_detect frontalface sf=1.1 scales 1..4 step=2, 3840x2160, batch %d per GPU" % n,
                "frames_per_gpu": n, "windows_per_frame": NWIN4,
                "l2": "integral tables (%.1f GiB per GPU) exceed the 126 MB L2" % (n * H4 * W4 * 4 / 2**30)}
    if wl == "c5":
        return {"workload": "c5: blur r=5 -> sobel -> orb_extract(nkps=1250,t=20) -> integral + lbp_detect(sf 1.1, scales 1..4, step 2), 1920x1080, %d frames per GPU" % n,
                "frames_per_gpu": n, "l2": "inputs (%.1f GiB per GPU) exceed the 126 MB L2" % (n * H3 * W3 / 2**30)}
    raise KeyError(wl)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


# ------------------------------------------------------------------ host cores
def host_cores():
    """cores this process may really use: the scheduler affinity, capped by the cgroup CPU quota
    (round 1's CPU arm sized its pool from the affinity alone and was 5.7x slower on a quota-limited box)"""
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:          # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-9))))
    try:
        load1 = os.getloadavg()[0]
    except Exception:
        load1 = None
    return cores, {"affinity": aff, "cgroup_quota_cores": quota, "loadavg_1m_at_start": load1}


def pin_to_gpu_numa(local):
    """keep this rank (and the pinned buffers it allocates) on the NUMA node of its GPU"""
    info = {"pinned": False}
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if len(bus.split(":")[0]) > 4:
            bus = bus[-12:]                                  # 00000000:1B:00.0 -> 0000:1b:00.0
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            txt = f.read().strip()
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            info["numa_node"] = int(f.read().strip())
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        before = os.sched_getaffinity(0)
        want = cpus & before
        if want:
            os.sched_setaffinity(0, want)
            info.update({"pinned": True, "cpus": len(want), "local_cpulist": txt})
        info["_restore"] = before
    except Exception as e:   # noqa: BLE001
        info["error"] = repr(e)[:120]
    return info


# ------------------------------------------------------------------ reference CPU arm
def _cpu_worker(args):
    """one process: run the real reference (or the oracle port) on `nframes` frames"""
    kind, workload, seed, nframes = args
    import numpy as np
    import _libs as L
    units = 0
    busy = 0.0
    if kind == "reference":
        R = L.ref()
    else:
        O = L.oracle()
    for i in range(nframes):
        rng = np.random.default_rng(seed * 1000 + i)
        if workload == "c2":
            a = rng.integers(0, 256, (H2, W2), dtype=np.uint8)
            b = np.empty_like(a); s = np.zeros_like(a)
            t0 = time.perf_counter()
            if kind == "reference":
                R.gs_blur(L.img(b), L.img(a), R2); R.gs_sobel(L.img(s), L.img(b))
            else:
                O.gso_blur(L.ptr(b), L.ptr(a), W2, H2, R2); O.gso_sobel(L.ptr(s), L.ptr(b), W2, H2)
            units += W2 * H2
        elif workload == "c3":
            a = L.natural_like(W3, H3, seed * 1000 + i)
            k = np.zeros(NK3, L.KP_DTYPE); sm = np.zeros_like(a)
            t0 = time.perf_counter()
            if kind == "reference":
                R.gs_orb_extract(L.img(a), L.ptr(k), NK3, T3, L.ptr(sm))
            else:
                O.gso_orb_extract(L.ptr(a), W3, H3, L.ptr(k), NK3, T3, L.ptr(sm))
            units += W3 * H3
        else:  # c4
            a = L.natural_like(W4, H4, seed * 1000 + i)
            ii = np.empty(a.shape, np.uint32); r = np.zeros(65536, L.RECT_DTYPE)
            cas = None if kind == "reference" else L.HostCascade()
            t0 = time.perf_counter()
            if kind == "reference":
                R.gs_integral(L.img(a), L.ptr(ii))
                R.gs_lbp_detect(R.ref_frontalface(), L.ptr(ii), W4, H4, L.ptr(r), 65536, 1.1, 1.0, 4.0, 2)
            else:
                O.gso_integral(L.ptr(a), W4, H4, L.ptr(ii))
                O.gso_lbp_detect(cas.ptr, L.ptr(ii), W4, H4, L.ptr(r), 65536, 1.1, 1.0, 4.0, 2)
            units += NWIN4
        busy += time.perf_counter() - t0
    return units, busy


def cpu_reference(workload, steps=1, warmup=0, max_cores=None, budget_s=150.0):
    """Frame-parallel over the host cores (one process per core: gs_orb_extract's static buffer is
    not thread-safe, reference grayskull.h:655).  A step = frames_per_core frames on every core at once;
    its time is the slowest core's.  First a single frame on ONE core (per-core throughput, and the
    calibration that keeps the whole arm inside `budget_s`).  Returns (value, dict)."""
    import _libs as L
    kind = "reference" if L.have_ref() else "port"
    if kind == "port":
        L.oracle()
    cores, core_info = host_cores()
    if max_cores:
        cores = min(cores, max_cores)
    fpc = {"c2": 1, "c3": 4, "c4": 1}[workload]
    scale = 1e-6 if workload in ("c2", "c3") else 1.0
    unit_name = "Mpixels/s" if workload in ("c2", "c3") else "windows/s"
    ctx = mp.get_context("fork")
    t_begin = time.perf_counter()
    with ctx.Pool(cores) as pool:
        u1, t1 = pool.apply(_cpu_worker, ((kind, workload, 9999, 1),))     # one frame, one core, idle box
        per_core = u1 / t1 * scale
        # predicted step time if the cores really run in parallel; shrink the plan to the budget
        step_pred = t1 * fpc * 1.3
        total = warmup + steps
        fit = max(1, int((budget_s - t1) / max(step_pred, 1e-3)))
        run_warm = min(warmup, max(0, fit - 1)) if fit < total else warmup
        run_steps = max(1, min(steps, fit - run_warm))
        per_step = []
        for s in range(run_warm + run_steps):
            res = pool.map(_cpu_worker, [(kind, workload, s * 64 + c, fpc) for c in range(cores)])
            if s >= run_warm:   # all cores run concurrently: the step takes as long as the slowest one
                per_step.append((sum(u for u, _ in res), max(t for _, t in res)))
            spent = time.perf_counter() - t_begin
            left = run_warm + run_steps - (s + 1)
            if per_step and left and spent + spent / (s + 1) > budget_s * 1.15:
                break              # the box is slower than the calibration said (quota / neighbours): stop early
    units = sum(u for u, _ in per_step)
    secs = sum(t for _, t in per_step)
    value = units / secs * scale
    what = {"c2": "4096x4096, gs_blur r=5 + gs_sobel", "c3": "1920x1080, gs_orb_extract nkps=1250 t=20",
            "c4": "3840x2160, gs_integral + gs_lbp_detect"}[workload]
    info = {"value": value, "unit": unit_name, "cores": cores, "kind": kind,
            "sample": "%d frames of %s per step (%d per core, one process per core; gcc -std=c99 -O2)" % (cores * fpc, what, fpc),
            "per_core": per_core, "per_core_sample": "1 frame on 1 core before the pool starts",
            "parallel_efficiency": value / (per_core * cores) if per_core > 0 else None,
            "ms_per_step": 1e3 * secs / max(len(per_step), 1), "steps_run": len(per_step), "warmup_run": run_warm,
            "frames_per_step": cores * fpc, "host": core_info}
    return value, info


# ------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        t0 = time.time()
        while self.p is not None and time.time() - t0 < 3.0:     # first sample lands before timing starts
            if os.path.getsize(self.f.name) > 0:
                break
            time.sleep(0.01)

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, pw = [], 0, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, cmax, power = float(parts[0]), float(parts[1]), float(parts[2])
            except ValueError:
                continue
            mx = max(mx, cmax)
            sm.append(clk); pw.append(power)
            for nme, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "power_w": statistics.median(pw) if pw else None, "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------ GPU arm
class Ctx:
    """rank / device / timing plumbing shared by every measurement of the GPU arm"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        import grayskull_b200 as g
        self.torch, self.dist, self.g = torch, dist, g
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.numa = pin_to_gpu_numa(self.local)
        torch.cuda.set_device(self.local)
        self.lib = g.lib()
        g._lib.check(self.lib.gs_b200_set_device(self.local), "set_device")
        self.dev = torch.device("cuda", self.local)
        self.group_ready = False
        if self.world > 1:
            self.init_group()
        self.hbm, self.peak_kind = peaks()

    def init_group(self):
        # NCCL may print a version banner on stdout (NCCL_DEBUG=VERSION): keep stdout for the ONE json line
        if self.group_ready:
            return
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            if self.world > 1:
                self.dist.init_process_group("nccl", device_id=self.dev)
            else:   # N = 1: a one-rank NCCL group so that the `shard` section runs the same code path
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                os.environ.setdefault("MASTER_PORT", str(29700 + os.getpid() % 200))
                self.dist.init_process_group("nccl", rank=0, world_size=1, device_id=self.dev)
            self.dist.barrier()            # forces communicator creation now
            self.torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
        self.group_ready = True

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world > 1:
            t = self.torch.tensor([float(v)], device=self.dev, dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return float(v)

    def time_steps(self, fn, steps, warmup, clocks=None):
        """W warm-ups, then K steps between barrier+sync, CUDA events on the launching stream, max over ranks.
        clocks: list that receives the nvidia-smi sample of the timed region (rank 0)"""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        sampler = ClockSampler(self.local) if (clocks is not None and self.rank == 0) else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        if sampler:
            clocks.append(sampler.stop())
        return self.max_over_ranks(e0.elapsed_time(e1))

    def kernel_table(self, kernels, steps):
        """per-entry-point CUDA-event time (each timed alone, back to back, inputs larger than L2)"""
        kres = {}
        for name, (fn, algo_bytes) in kernels.items():
            ksteps = max(min(steps, 100) // 2, 5)
            kms = self.time_steps(fn, ksteps, 3) / ksteps
            gbs = algo_bytes / (kms * 1e-3) / 1e9
            kres[name] = {"ms": kms, "algorithmic_bytes": algo_bytes, "achieved_gbs": gbs, "frac": gbs / self.hbm}
        return kres

    def roofline(self, kres, wl, n):
        dom = max(kres, key=lambda k: kres[k]["ms"])
        r = {"kernel": dom, "bound": "hbm", "achieved": kres[dom]["achieved_gbs"], "peak": self.hbm,
             "peak_source": self.peak_kind + (" (MEASURED_PEAKS.json hbm_gbs)" if self.peak_kind == "measured" else " (B200_PROFILING.md)"),
             "unit": "GB/s", "frac": kres[dom]["frac"], "traffic": None,
             "algorithmic_bytes_per_launch": kres[dom]["algorithmic_bytes"], "ms_per_launch": kres[dom]["ms"]}
        try:
            # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this entry point.
            # `traffic` is filled only when the capture was taken at THIS batch size; a capture at another batch
            # is reported per frame under traffic_profiled (dirty lines still in L2 at kernel end make small
            # batches under-report the writes).
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                t = json.load(f).get(wl, {}).get(dom)
            if t:
                if int(t.get("batch", 0)) == int(n):
                    r["traffic"] = t["dram_bytes_per_frame"] * n
                    r["traffic_source"] = t.get("source")
                else:
                    r["traffic_profiled"] = {"dram_bytes_per_frame": t["dram_bytes_per_frame"], "batch": t.get("batch"),
                                             "scaled_to_this_launch": t["dram_bytes_per_frame"] * n, "source": t.get("source")}
        except Exception:
            pass
        return r


def build_workload(cx, wl, batch):
    """-> dict(step, units_per_step, kernels, cfg, launches hint, keepalive tensors)"""
    torch, api, g, dev = cx.torch, __import__("grayskull_b200.api", fromlist=["api"]), cx.g, cx.dev
    torch.manual_seed(1234 + cx.rank)
    W = {}
    if wl == "c2":
        n, h, w = batch or B2, H2, W2
        src = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        blur = torch.empty_like(src)
        sob = torch.zeros_like(src)
        fused = hasattr(api, "blur_sobel_batch")

        def step_unfused():
            api.blur_batch(src, R2, out=blur)
            api.sobel_batch(blur, out=sob)

        def step_fused():
            api.blur_sobel_batch(src, R2, out=sob)

        # Headline = the two per-op kernels, BASELINE configs[1] read literally.  The one-pass gs_b200_blur_sobel_batch
        # (2 B/px of HBM traffic instead of 4) is measured next to it: it is instruction-bound (22 lane-instr/px against
        # 18.4 for the pair, DESIGN.md section 3) and slower on this machine, so it does not carry the headline.
        W.update(step=step_unfused, variants={"unfused": step_unfused}, fused=False)
        if fused:
            W["variants"]["fused"] = step_fused
        px = float(n * h * w)
        W["kernels"] = {"gs_blur_r5": (lambda: api.blur_batch(src, R2, out=blur), 2.0 * px),
                        "gs_sobel": (lambda: api.sobel_batch(blur, out=sob), px + 1.0 * n * (h - 2) * (w - 2))}
        if fused:
            W["variant_kernels"] = {"gs_blur_sobel_r5": (step_fused, px + 1.0 * n * (h - 2) * (w - 2))}
        W.update(units=n * h * w, n=n, h=h, w=w, src=src, keep=(blur, sob), outputs=lambda: {"blur": blur, "sobel": sob})
    elif wl == "c3":
        n, h, w = batch or B3, H3, W3
        noise = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        src = api.blur_batch(noise, 3)      # "blurred noise": natural-image-like autocorrelation
        del noise
        sm = torch.zeros_like(src)
        kps = torch.empty((n, NK3, 12), dtype=torch.int32, device=dev)
        cnt = torch.zeros((n,), dtype=torch.int32, device=dev)
        st = api._stream

        def step():
            g._lib.check(cx.lib.gs_b200_orb_extract_batch(api._p(src), w, h, n, api._p(sm), api._p(kps), api._p(cnt),
                                                          NK3, T3, st()), "orb_extract_batch")

        W.update(step=step, kernels={"gs_orb_extract": (step, 2.0 * n * h * w + 48.0 * n * NK3)},
                 units=n * h * w, n=n, h=h, w=w, src=src, keep=(sm, kps, cnt),
                 outputs=lambda: {"scoremap": sm, "keypoints": _keypoints(kps, cnt), "keypoint_counts": cnt})
    elif wl == "c4":
        n, h, w = batch or B4, H4, W4
        cas = g.load_cascade()
        noise = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        src = api.blur_batch(noise, 3)
        del noise
        ii = torch.empty((n, h, w), dtype=torch.int32, device=dev)
        rects = torch.empty((n, 65536, 4), dtype=torch.int32, device=dev)
        rc = torch.zeros((n,), dtype=torch.int32, device=dev)
        nwin = api.lbp_window_count(cas, w, h, 1.1, 1.0, 4.0, 2)
        assert (w, h) != (W4, H4) or nwin == NWIN4
        st = api._stream

        def lbp():
            g._lib.check(cx.lib.gs_b200_lbp_detect_batch(cas.ptr, api._p(ii), w, h, n, api._p(rects), api._p(rc), 65536,
                                                         1.1, 1.0, 4.0, 2, st()), "lbp_detect_batch")

        def step():
            api.integral_batch(src, out=ii)
            lbp()

        W.update(step=step, kernels={"gs_integral": (lambda: api.integral_batch(src, out=ii), 5.0 * n * h * w),
                                     "gs_lbp_detect": (lbp, 4.0 * n * h * w)},
                 units=n * nwin, n=n, h=h, w=w, src=src, keep=(ii, rects, rc, cas), nwin=nwin,
                 outputs=lambda: {"integral": ii, "rects": _valid_rows(rects, rc), "rect_counts": rc}, unsigned={"integral"})
    elif wl == "c5":
        # BASELINE configs[4]: blur -> sobel -> FAST/ORB -> integral + LBP on 1920x1080 frames, sharded by frame
        # (8192 frames over 8 GPUs = 1024 per GPU).  FAST and LBP both run on the sobel output (SURVEY.md 8d).
        from grayskull_b200 import pipeline
        n, h, w = batch or 256, H3, W3
        cas = g.load_cascade()
        src = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        pipe = pipeline.FramePipeline(cas, n, h, w, dev)
        up = pipe

        def step():
            pipe.run(src, 0)

        st = api._stream
        P = pipe.p
        px = float(n * h * w)
        kern = {"gs_blur_r5": (lambda: api.blur_batch(src, R2, out=up.blur if up.blur is not None else pipe.score), 2.0 * px),
                "gs_sobel": (lambda: api.sobel_batch(src, out=pipe.score), 2.0 * px),
                "gs_orb_extract": (lambda: g._lib.check(cx.lib.gs_b200_orb_extract_batch(
                    api._p(pipe.sobel), w, h, n, api._p(pipe.score), api._p(pipe.kps), api._p(pipe.kcounts), P["nkps"],
                    P["threshold"], st())), 2.0 * px),
                "gs_integral": (lambda: api.integral_batch(pipe.sobel, out=pipe.ii), 5.0 * px),
                "gs_lbp_detect": (lambda: g._lib.check(cx.lib.gs_b200_lbp_detect_batch(
                    cas.ptr, api._p(pipe.ii), w, h, n, api._p(pipe.rects), api._p(pipe.rcounts), P["max_rects"],
                    P["scale_factor"], P["min_scale"], P["max_scale"], P["step"], st())), 4.0 * px)}
        if hasattr(api, "blur_sobel_batch"):
            W["variant_kernels"] = {"gs_blur_sobel_r5": (lambda: api.blur_sobel_batch(src, R2, out=pipe.score), 2.0 * px)}
        W.update(step=step, kernels=kern, units=n * h * w, n=n, h=h, w=w, src=src, keep=(pipe, up, cas),
                 outputs=lambda: {"sobel": pipe.sobel, "keypoints": _keypoints(pipe.kps, pipe.kcounts),
                                  "keypoint_counts": pipe.kcounts, "rects": _valid_rows(pipe.rects, pipe.rcounts),
                                  "rect_counts": pipe.rcounts})
    elif wl == "match":
        # SURVEY.md 8(f) N1: gs_match_orb over frame pairs (1250 x 1250 descriptors each, the c3 keypoint budget).
        # Not HBM-bound: 8 POPC per descriptor comparison on the 16-lane/clk/SM POPC path bounds it.
        npairs, nd = batch or 2048, NK3
        gen = torch.Generator(device=dev); gen.manual_seed(77 + cx.rank)
        k2 = torch.randint(-2**31, 2**31 - 1, (npairs, nd, 12), dtype=torch.int32, device=dev, generator=gen)
        k1 = k2[:, torch.randperm(nd, device=dev)].clone()
        flip = (torch.rand((npairs, nd, 8), device=dev, generator=gen) < 0.6).to(torch.int32) << torch.randint(0, 31, (npairs, nd, 8), device=dev, generator=gen).to(torch.int32)
        k1[:, :, 4:] ^= flip                     # near-duplicates: ~5 flipped bits per descriptor
        k1[:, nd // 2:, 4:] = torch.randint(-2**31, 2**31 - 1, (npairs, nd - nd // 2, 8), dtype=torch.int32, device=dev, generator=gen)
        del flip
        cnt = torch.full((npairs,), nd, dtype=torch.int32, device=dev)
        last = {}

        def step():
            last["matches"], last["counts"] = api.match_orb_batch(k1, cnt, k2, cnt, nd, 60.0)

        W.update(step=step, kernels={"gs_match_orb": (step, 2.0 * npairs * nd * 48 + 12.0 * npairs * nd)},
                 units=npairs * nd * nd, n=npairs, h=nd, w=nd, src=k1, keep=(k2, cnt),
                 outputs=lambda: {"matches": _valid_rows(last["matches"], last["counts"]), "match_counts": last["counts"]},
                 metric=("256-bit descriptor comparisons/s, gs_match_orb 1250 x 1250 per frame pair", "Gcomparisons/s", 1e-9),
                 cfg={"workload": "match: gs_match_orb max_distance=60, 1250 x 1250 descriptors per pair, %d pairs per GPU" % npairs,
                      "pairs_per_gpu": npairs, "l2": "descriptor sets (%.0f MB per GPU) exceed the 126 MB L2" % (2 * npairs * nd * 48 / 1e6)})
    elif wl == "tmatch":
        # SURVEY.md 8(f) N3: gs_match_template, one 32x32 template against 1920x1080 frames (compute-bound:
        # 11 instructions per 16 squared differences)
        n, h, w = batch or 16, H3, W3
        tw = th = 32
        noise = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        src = api.blur_batch(noise, 2)
        del noise
        tmpl = src[0, 500:500 + th, 900:900 + tw].contiguous()
        res = torch.empty((n, h - th + 1, w - tw + 1), dtype=torch.uint8, device=dev)
        last = {}

        def step():
            api.match_template_batch(src, tmpl, out=res)
            last["best"] = api.find_best_match_batch(res)

        W.update(step=step, kernels={"gs_match_template": (lambda: api.match_template_batch(src, tmpl, out=res), 2.0 * n * h * w)},
                 units=n * (h - th + 1) * (w - tw + 1) * tw * th, n=n, h=h, w=w, src=src, keep=(tmpl, res),
                 outputs=lambda: {"match": res, "best_match": last["best"]},
                 metric=("squared differences/s, gs_match_template 32x32 template, 1920x1080 uint8", "Gtaps/s", 1e-9),
                 cfg={"workload": "tmatch: gs_match_template + gs_find_best_match, 32x32 template, 1920x1080, batch %d per GPU" % n,
                      "frames_per_gpu": n, "l2": "compute-bound; frames (%.0f MB per GPU) stream through L2" % (n * h * w / 1e6)})
    elif wl == "ops":
        # per-op table (every stencil / resampling op of the path at 4096x4096), not a driver line
        import numpy as np
        n, h, w = batch or 64, H2, W2
        src = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, device=dev)
        out = torch.zeros_like(src)
        half = torch.empty((n, h // 2, w // 2), dtype=torch.uint8, device=dev)
        odd = torch.empty((n, 1440, 2560), dtype=torch.uint8, device=dev)
        ii = torch.empty((n, h, w), dtype=torch.int32, device=dev)
        hist = torch.empty((n, 256), dtype=torch.int32, device=dev)
        K_SHARPEN = np.array([[0, -1, 0], [-1, 5, -1], [0, -1, 0]], np.int8)
        K_GAUSS = np.array([[1, 2, 1], [2, 4, 2], [1, 2, 1]], np.int8)
        oth = torch.empty((n,), dtype=torch.uint8, device=dev)
        px = float(n * h * w)
        kernels = {
            "gs_sobel": (lambda: api.sobel_batch(src, out=out), 2.0 * px),
            "gs_erode": (lambda: api.erode_batch(src, out=out), 2.0 * px),
            "gs_dilate": (lambda: api.dilate_batch(src, out=out), 2.0 * px),
            "gs_blur_r1": (lambda: api.blur_batch(src, 1, out=out), 2.0 * px),
            "gs_blur_r3": (lambda: api.blur_batch(src, 3, out=out), 2.0 * px),
            "gs_blur_r5": (lambda: api.blur_batch(src, 5, out=out), 2.0 * px),
            "gs_blur_r7": (lambda: api.blur_batch(src, 7, out=out), 2.0 * px),
            "gs_blur_r9": (lambda: api.blur_batch(src, 9, out=out), 2.0 * px),
            "gs_blur_r15": (lambda: api.blur_batch(src, 15, out=out), 2.0 * px),
            "gs_blur_r31": (lambda: api.blur_batch(src, 31, out=out), 2.0 * px),
            "gs_adaptive_threshold_r5": (lambda: api.adaptive_threshold_batch(src, 5, 2, out=out), 2.0 * px),
            "gs_adaptive_threshold_r15": (lambda: api.adaptive_threshold_batch(src, 15, 5, out=out), 2.0 * px),
            "gs_downsample": (lambda: api.downsample_batch(src, out=half), 1.25 * px),
            "gs_resize_to_half": (lambda: api.resize_batch(src, w // 2, h // 2, out=half), 1.25 * px),
            "gs_resize_to_2560x1440": (lambda: api.resize_batch(src, 2560, 1440, out=odd), px + n * 2560.0 * 1440.0),
            "gs_integral": (lambda: api.integral_batch(src, out=ii), 5.0 * px),
            "gs_filter_sharpen": (lambda: api.filter_batch(src, K_SHARPEN, 1, out=out), 2.0 * px),
            "gs_filter_gaussian": (lambda: api.filter_batch(src, K_GAUSS, 16, out=out), 2.0 * px),
            "gs_histogram": (lambda: api.histogram_batch(src, out=hist), 1.0 * px),
            "gs_otsu_threshold": (lambda: api.otsu_threshold_batch(src, hist=hist, out=oth), 1.0 * px),
            "gs_threshold": (lambda: api.threshold_batch(out, 128), 2.0 * px),
        }
        if hasattr(api, "blur_sobel_batch"):
            kernels["gs_blur_sobel_r5"] = (lambda: api.blur_sobel_batch(src, 5, out=out), 2.0 * px)

        def step():
            for fn, _ in kernels.values():
                fn()

        W.update(step=step, kernels=kernels, units=n * h * w * len(kernels), n=n, h=h, w=w, src=src,
                 keep=(out, half, odd, ii, hist, oth),
                 outputs=lambda: {"out": out, "half": half, "resized_2560x1440": odd, "integral": ii, "histogram": hist,
                                  "otsu": oth}, unsigned={"integral"},
                 metric=("Mpixels/s summed over the per-op table, 4096x4096 uint8", "Mpixels/s", 1e-6),
                 cfg={"workload": "ops: every stencil/resampling op once, 4096x4096 synthetic uint8, batch %d per GPU" % n,
                      "frames_per_gpu": n, "l2": "inputs (%.1f GiB per GPU) exceed the 126 MB L2" % (n * h * w / 2**30)})
    else:
        raise SystemExit("unknown workload " + wl)
    if "metric" not in W:
        W["metric"] = METRICS[wl]
        W["cfg"] = workload_cfg(wl, W["n"])
    return W


def _u32(t):
    """int32-typed storage of unsigned 32-bit words -> their values as int64"""
    import torch
    return t.to(torch.int64) & 0xFFFFFFFF


def _valid_rows(t, counts):
    """(n, cap, k) records of which counts[i] are valid in frame i: the rows past the count zeroed (they hold
    whatever an earlier step or allocation left there)"""
    import torch
    keep = torch.arange(t.shape[1], device=t.device)[None, :] < counts[:, None].to(torch.int64)
    return t * keep[..., None].to(t.dtype)


def _keypoints(kps, counts):
    """(n, nkps, 12) struct gs_keypoint words -> x, y, response, angle, descriptor[8] as values (float64)"""
    import torch
    k = _valid_rows(kps, counts)
    v = _u32(k).to(torch.float64)
    v[..., 3] = k[..., 3].contiguous().view(torch.float32).to(torch.float64)
    return v


def dump_outputs(outputs, out_dir, unsigned=()):
    """write each output as out_dir/<name>.npy (see the module docstring for dtypes and sampling).
    unsigned: names of int32-typed outputs that hold unsigned 32-bit words"""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    left, names = DUMP_BYTES, sorted(outputs, key=lambda n: outputs[n].numel())
    for i, name in enumerate(names):
        t = outputs[name]
        dt = torch.float32 if t.element_size() <= 2 or t.dtype == torch.float32 else torch.float64
        size = 4 if dt == torch.float32 else 8
        k = min(t.numel(), left // (len(names) - i) // size)
        if t.numel() > k:                        # sample first: only the k picked values are widened
            idx = np.sort(np.random.default_rng(0).integers(0, t.numel(), k))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        if name in unsigned:
            t = _u32(t)
        np.save(os.path.join(out_dir, name + ".npy"), t.to(dt).cpu().numpy())
        left -= k * size


def measure(cx, wl, batch, steps, warmup, with_kernels=True, dump=None):
    """headline numbers of one workload: device-resident steps, per-entry-point table, roofline, clocks.
    dump: directory for the outputs of the last timed step (written before anything else reuses the buffers)"""
    W = build_workload(cx, wl, batch)
    metric, unit, scale = W["metric"]
    clocks = []
    l0 = cx.lib.gs_b200_launch_count()
    ms = cx.time_steps(W["step"], steps, warmup, clocks=clocks)
    launched = cx.lib.gs_b200_launch_count() - l0
    if dump and cx.rank == 0:
        dump_outputs(W["outputs"](), dump, W.get("unsigned", ()))
    out = {"metric": metric, "value": W["units"] * cx.world * steps / (ms * 1e-3) * scale, "unit": unit,
           "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "config": W["cfg"],
           "clocks": clocks[0] if clocks else None,
           "gpu_launches": int(launched * steps // (steps + warmup)), "launches_per_step": int(launched // (steps + warmup))}
    if "variants" in W and len(W["variants"]) > 1:
        v = {}
        for name, fn in W["variants"].items():
            vs = max(5, min(steps, 50))
            v[name] = cx.time_steps(fn, vs, 3) / vs
        out["ms_per_step_variants"] = v
        out["headline_variant"] = "fused" if W.get("fused") else "unfused"
    if with_kernels:
        kres = cx.kernel_table(W["kernels"], steps)
        out["roofline"] = cx.roofline(kres, wl, W["n"])      # dominant kernel OF THE HEADLINE STEP
        if "variant_kernels" in W:
            kres.update({k + " (variant, not in the step)": v for k, v in cx.kernel_table(W["variant_kernels"], steps).items()})
        out["kernels"] = kres
    return out, W


def e2e_c2(cx, W, args):
    """c2 through the C ABI with HOST buffers, copies inside the timed region (wall clock, max over ranks)"""
    torch, lib, g = cx.torch, cx.lib, cx.g
    n, h, w, src = W["n"], W["h"], W["w"], W["src"]
    scale = 1e-6
    ne = min(n, args.e2e_frames)
    chunk, nstreams = args.e2e_chunk, args.e2e_streams
    hin = torch.empty((ne, h, w), dtype=torch.uint8).pin_memory()
    hout = torch.empty((ne, h, w), dtype=torch.uint8).pin_memory()
    hin.copy_(src[:ne].cpu())
    streams = [torch.cuda.Stream(device=cx.dev) for _ in range(nstreams)]
    fused = W.get("fused")
    dbuf = [(torch.empty((chunk, h, w), dtype=torch.uint8, device=cx.dev), torch.empty((chunk, h, w), dtype=torch.uint8, device=cx.dev),
             torch.zeros((chunk, h, w), dtype=torch.uint8, device=cx.dev)) for _ in range(nstreams)]

    def e2e_step():
        for ci, lo in enumerate(range(0, ne, chunk)):
            st = streams[ci % nstreams]
            a, b, c = dbuf[ci % nstreams]
            sp = C.c_void_p(st.cuda_stream)
            k = min(chunk, ne - lo)
            g._lib.check(lib.gs_b200_memcpy_h2d(C.c_void_p(a.data_ptr()), C.c_void_p(hin[lo].data_ptr()), k * h * w, sp))
            if fused:
                g._lib.check(lib.gs_b200_blur_sobel_batch(C.c_void_p(c.data_ptr()), C.c_void_p(a.data_ptr()), w, h, k, R2, sp))
            else:
                g._lib.check(lib.gs_b200_blur_batch(C.c_void_p(b.data_ptr()), C.c_void_p(a.data_ptr()), w, h, k, R2, sp))
                g._lib.check(lib.gs_b200_sobel_batch(C.c_void_p(c.data_ptr()), C.c_void_p(b.data_ptr()), w, h, k, sp))
            g._lib.check(lib.gs_b200_memcpy_d2h(C.c_void_p(hout[lo].data_ptr()), C.c_void_p(c.data_ptr()), k * h * w, sp))
        for st in streams:
            st.synchronize()

    for _ in range(2):
        e2e_step()
    cx.barrier()
    t0 = time.perf_counter()
    ksteps = max(3, min(args.steps, 100) // 10)
    for _ in range(ksteps):
        e2e_step()
    cx.barrier()
    dt = cx.max_over_ranks(time.perf_counter() - t0)
    e2e = {"value": ne * h * w * cx.world * ksteps / dt * scale, "unit": "Mpixels/s", "h2d_bytes_per_step": ne * h * w,
           "d2h_bytes_per_step": ne * h * w, "frames_per_step": ne, "steps": ksteps,
           "pcie_gbs_each_way": ne * h * w * ksteps / dt / 1e9,
           "path": "pinned host -> gs_b200_memcpy_h2d -> %s -> gs_b200_memcpy_d2h, %d-frame chunks on %d streams" % (
               "gs_b200_blur_sobel_batch" if fused else "gs_b200_blur_batch -> gs_b200_sobel_batch", chunk, nstreams),
           "numa": {k: v for k, v in cx.numa.items() if not k.startswith("_")}}
    del hin, hout, dbuf

    # the reference's own call shape: one image per call, plain (pageable) host pointers, synchronous
    import numpy as np
    nd = min(8, ne)
    fr = [src[i].cpu().numpy() for i in range(nd)]
    tmp = [np.empty_like(fr[0]) for _ in range(nd)]
    outs = [np.zeros_like(fr[0]) for _ in range(nd)]
    Img = g._lib.Image

    def dropin_step():
        for i in range(nd):
            lib.gs_blur(Img(w, h, tmp[i].ctypes.data), Img(w, h, fr[i].ctypes.data), R2)
            lib.gs_sobel(Img(w, h, outs[i].ctypes.data), Img(w, h, tmp[i].ctypes.data))

    dropin_step()
    cx.barrier()
    t0 = time.perf_counter()
    dsteps = 3
    for _ in range(dsteps):
        dropin_step()
    cx.barrier()
    dt = cx.max_over_ranks(time.perf_counter() - t0)
    dropin = {"value": nd * h * w * cx.world * dsteps / dt * scale, "unit": "Mpixels/s", "frames_per_step": nd, "steps": dsteps,
              "h2d_bytes_per_step": 2 * nd * h * w, "d2h_bytes_per_step": nd * h * w + nd * (h - 2) * (w - 2),
              "path": "gs_blur(dst, src, 5) then gs_sobel(dst, src) per frame with pageable host pointers (the reference's call "
                      "shape, include/grayskull.h): each call stages its image in and out and synchronises; the blurred "
                      "intermediate crosses PCIe twice; sobel copies back only the interior so that dst keeps its border bytes"}
    return e2e, dropin


def shard_section(cx, args):
    """BASELINE configs[4] / SURVEY.md 8(e): rank 0 holds every frame; ONE scatter of uint8 frames (grouped
    ncclSend/ncclRecv), the c5 frame pipeline on every rank's shard, ONE gather of sobel maps + keypoints + rects.
    Reported including and excluding the two collectives, whole-shard and chunk-overlapped."""
    torch, g = cx.torch, cx.g
    from grayskull_b200 import pipeline, shard
    cx.init_group()
    per = args.shard_frames
    n_total, h, w = per * cx.world, H3, W3
    cas = g.load_cascade()
    root = None
    if cx.rank == 0:
        root = torch.empty((n_total, h, w), dtype=torch.uint8, device=cx.dev)
        for lo in range(0, n_total, 256):                      # generate in slices: randint's int64 temp is 8 B/px
            hi = min(n_total, lo + 256)
            root[lo:hi] = torch.randint(0, 256, (hi - lo, h, w), dtype=torch.uint8, device=cx.dev)
    lo, hi = shard.shard_range(n_total, cx.rank, cx.world)
    pipe = pipeline.FramePipeline(cas, hi - lo, h, w, cx.dev)
    run = shard.ShardedRun(pipe, n_total, h, w, cx.dev)
    steps = max(1, args.shard_steps)

    def serial():
        return run.run_serial(root)

    serial()                                                   # warm-up (workspaces, NCCL channels)
    cx.barrier()
    acc = {"scatter": 0.0, "compute": 0.0, "gather": 0.0, "total": 0.0}
    clocks = []
    sampler = ClockSampler(cx.local) if cx.rank == 0 else None
    for _ in range(steps):
        cx.barrier()
        ev = serial()
        cx.barrier()
        acc["scatter"] += cx.max_over_ranks(ev[0].elapsed_time(ev[1]))
        acc["compute"] += cx.max_over_ranks(ev[1].elapsed_time(ev[2]))
        acc["gather"] += cx.max_over_ranks(ev[2].elapsed_time(ev[3]))
        acc["total"] += cx.max_over_ranks(ev[0].elapsed_time(ev[3]))
    if sampler:
        clocks.append(sampler.stop())
    ms = {k: v / steps for k, v in acc.items()}
    nch = max(1, args.shard_chunks)
    run.run_overlapped(root, nch)                              # warm-up of the chunked form
    cx.barrier()
    ov = 0.0
    for _ in range(steps):
        cx.barrier()
        e0, e1 = run.run_overlapped(root, nch)
        cx.barrier()
        ov += cx.max_over_ranks(e0.elapsed_time(e1))
    ov /= steps
    bs, bg = run.bytes_scattered(), run.bytes_gathered()
    px = float(n_total) * h * w
    out = {"workload": workload_cfg("c5", per)["workload"], "frames_total": n_total, "frames_per_gpu": per, "steps": steps,
           "collective": "grouped ncclSend/ncclRecv from / to rank 0 (torch.distributed batch_isend_irecv); nothing else crosses ranks",
           "bytes_scattered": bs, "bytes_gathered": bg,
           "ms": ms,
           "scatter_gbs": bs / (ms["scatter"] * 1e-3) / 1e9 if bs else None,
           "gather_gbs": bg / (ms["gather"] * 1e-3) / 1e9 if bg else None,
           "root_link_bound_gbs": NVLINK_GBS,
           "scatter_frac_of_link": (bs / (ms["scatter"] * 1e-3) / 1e9 / NVLINK_GBS) if bs else None,
           "gather_frac_of_link": (bg / (ms["gather"] * 1e-3) / 1e9 / NVLINK_GBS) if bg else None,
           "mpix_s_excluding_collectives": px / (ms["compute"] * 1e-3) * 1e-6,
           "mpix_s_including_collectives": px / (ms["total"] * 1e-3) * 1e-6,
           "overlapped": {"chunks": nch, "ms": ov, "mpix_s": px / (ov * 1e-3) * 1e-6,
                          "how": "every rank's shard in %d pieces; piece c of all ranks is one NCCL group on a side stream, "
                                 "scattered while piece c-1 is processed and gathered while piece c+1 is processed" % nch},
           "limit": None, "clocks": clocks[0] if clocks else None}
    comm = ms["scatter"] + ms["gather"]
    out["limit"] = ("pipeline compute (gs_lbp_detect) -- the two collectives are %.1f %% of the serial step" % (100.0 * comm / ms["total"])
                    if comm < ms["compute"] else "root NVLink egress / ingress (collectives are %.1f %% of the serial step)" % (100.0 * comm / ms["total"]))
    del run, pipe, root
    torch.cuda.empty_cache()
    return out


def gpu_main(args):
    cx = Ctx()
    torch = cx.torch
    wl = args.workload
    res, W = measure(cx, wl, args.batch, args.steps, args.warmup, dump=args.dump_outputs)
    metric, unit, scale = W["metric"]
    out = {"metric": res["metric"], "value": res["value"], "unit": unit, "n_gpus": cx.world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": {"c4": "u32", "match": "u32 (xor + popc)"}.get(wl, "u8"),
           "data": "synthetic (uniform iid u8, torch.randint; c3/c4: gs_blur r=3 of it)", "config": res["config"],
           "clocks": res["clocks"], "e2e": None, "gpu_launches": res["gpu_launches"],
           "launches_per_step": res["launches_per_step"], "roofline": res["roofline"], "kernels": res["kernels"],
           "cpu_baseline": None, "tma_path": bool(cx.lib.gs_b200_uses_tma(W["w"], W["h"], W["src"].data_ptr()))}
    for k in ("ms_per_step_variants", "headline_variant"):
        if k in res:
            out[k] = res[k]
    if wl == "c2" and not args.no_e2e:
        out["e2e"], out["e2e_dropin"] = e2e_c2(cx, W, args)
    del W
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, in the same run (default line only) ----
    cfgs = {}
    if wl == "c2" and not args.no_configs:
        for name, st, wu in (("c3", 20, 5), ("c4", 3, 1)):
            r, Wc = measure(cx, name, 0, st, wu)
            r["dtype"] = "u32" if name == "c4" else "u8"
            cfgs[name] = r
            del Wc
            torch.cuda.empty_cache()
        out["configs"] = cfgs
    if (wl == "c2" and not args.no_shard) or args.shard:
        out["shard"] = shard_section(cx, args)

    # ---- CPU baselines (rank 0, N == 1 only): the reference's C code on the host cores ----
    if "_restore" in cx.numa:
        try:
            os.sched_setaffinity(0, cx.numa["_restore"])
        except Exception:
            pass
    if cx.rank == 0 and cx.world == 1 and not args.no_cpu:
        if wl in ("c2", "c3", "c4"):
            _, out["cpu_baseline"] = cpu_reference(wl, steps=1, warmup=0, max_cores=args.cpu_cores or None, budget_s=40.0)
        for name in cfgs:
            _, cfgs[name]["cpu_baseline"] = cpu_reference(name, steps=1, warmup=0, max_cores=args.cpu_cores or None, budget_s=40.0)
        if wl == "match":
            import numpy as np
            import _libs as L
            from grayskull_b200 import api
            kind = "reference" if L.have_ref() else "port"
            fn = L.ref().gs_match_orb if kind == "reference" else L.oracle().gso_match_orb
            Wm = build_workload(cx, "match", 1)
            nd = NK3
            a = api.kps_to_numpy(Wm["src"][:1], Wm["keep"][1][:1])[0]; b = api.kps_to_numpy(Wm["keep"][0][:1], Wm["keep"][1][:1])[0]
            m = np.zeros(nd, L.MATCH_DTYPE)
            t0 = time.perf_counter(); reps = 0
            while time.perf_counter() - t0 < 5.0:
                fn(L.ptr(a), nd, L.ptr(b), nd, L.ptr(m), nd, 60.0); reps += 1
            dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": reps * nd * nd / dt * scale, "unit": unit, "cores": 1, "kind": kind,
                                   "sample": "%d calls of gs_match_orb on one 1250 x 1250 pair (gcc -std=c99 -O2, single thread)" % reps}

    if cx.rank == 0:
        print(json.dumps(out))
    if cx.group_ready:
        cx.dist.destroy_process_group()


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    value, cpu = cpu_reference(wl, steps=max(1, args.steps), warmup=max(0, args.warmup), budget_s=150.0)
    metric, unit, _ = METRICS[wl]
    nb = args.batch or {"c2": B2, "c3": B3, "c4": B4}[wl]
    out = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
           "steps": cpu["steps_run"], "warmup": cpu["warmup_run"], "ms_per_step": cpu["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8" if wl != "c4" else "u32",
           "data": "synthetic", "config": workload_cfg(wl, nb), "cpu_baseline": cpu,
           "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps (--impl reference: at most this many, see above)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5", "ops", "match", "tmatch"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU (default: the BASELINE config's batch)")
    ap.add_argument("--e2e-frames", type=int, default=64)
    ap.add_argument("--e2e-chunk", type=int, default=16)
    ap.add_argument("--e2e-streams", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the c3 / c4 objects of the default line")
    ap.add_argument("--no-shard", action="store_true", help="skip the scatter -> c5 -> gather section of the default line")
    ap.add_argument("--shard", action="store_true", help="add the shard section to a non-default workload's line")
    ap.add_argument("--shard-frames", type=int, default=B5, help="frames per GPU of the shard section (c5: 1024)")
    ap.add_argument("--shard-steps", type=int, default=2)
    ap.add_argument("--shard-chunks", type=int, default=4)
    ap.add_argument("--cpu-cores", type=int, default=0, help="cap the cores of the cpu_baseline sample (default: all)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "b200" or a.steps < 1):
        ap.error("--dump-outputs needs the GPU arm and --steps >= 1")
    if a.impl == "reference":
        reference_main(a)
    else:
        gpu_main(a)
