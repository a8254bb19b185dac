#!/usr/bin/env python
"""bench.py — fwd+bwd Msplats/s of the 2D-surfel rasterizer hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]

A "step" is one forward + one backward of the op (diff_surfel_rasterization.GaussianRasterizer as
/root/reference/gaussian_renderer/__init__.py:97-106 calls it, then autograd backward with dense
cotangents on all 10 output channels) over one synthetic view (SURVEY §8(d) generator).
Default workload = the configuration the metric is quoted on: 1 M surfels, 1920x1080, SH degree 3.
N > 1: one process per GPU (torchrun), independent views sharded one per rank, no data-path
collective ("scaling": "weak"); time = max over ranks.

Prints ONE JSON line (see the task contract): value (inputs resident in HBM), e2e (host buffers,
H2D of every input and D2H of outputs + gradients inside the timed region), roofline of the
dominant kernel (timed live with CUDA events on the launching stream), cpu_baseline (the C oracle
port on the host cores), clocks, gpu_launches.

--impl reference: the reference's CUDA rasterizer is not vendored in /root/reference (SURVEY §0), so
the reference arm is the CPU restatement (oracle/, "port") on the box's host cores, same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "2d-gaussian-splatting_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "fwd+bwd Msplats/sec at 1M surfels/1080p"
UNIT = "Msplats/s"


def workload_string(name, P, W, H):
    """config.workload: the same string in both arms."""
    return f"{name}: {P} surfels, {W}x{H}, SH degree 3, fwd+bwd, one view per GPU"


def algorithmic_bytes(P, V, R, W, H):
    """SURVEY §8(d) / BASELINE.md §2.3 per-stage algorithmic bytes."""
    N = W * H
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    return {
        "preprocess_fwd": 48 * P + 271 * V + 8 * P,
        "duplicate_with_keys": 20 * V + 12 * R,
        "sort": 24 * R,
        "identify_tile_ranges": 8 * R + 8 * tiles,
        "render_fwd": 76 * R + 60 * N,
        "render_bwd": 76 * R + 60 * N + 72 * R,
        "preprocess_bwd": 343 * V + 240 * V,
    }


DUMP_MAX_BYTES = 64 << 20
DUMP_PIXELS = 1 << 18          # image planes larger than this are written at this many pixels, ...
DUMP_SPLATS = 1 << 16          # ... per-splat arrays at this many splats


def _dump_sample(n, k, seed):
    """Sorted indices of a fixed, seeded sample of k out of n, or None when everything fits."""
    import numpy as np
    if n <= k:
        return None
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(out_dir, images, per_splat):
    """Writes one step's results as <out_dir>/<name>.npy (float32; sample indices float64).  images: name -> (C, H, W),
    per_splat: name -> (P, ...).  At large sizes the images are reduced to (C, DUMP_PIXELS) columns of the flattened
    H*W plane (pixel_index.npy) and the per-splat arrays to DUMP_SPLATS rows (splat_index.npy): the same indices
    whenever the shapes are the same, so that two builds can be compared output for output."""
    import numpy as np
    H, W = next(iter(images.values())).shape[1:]
    P = next(iter(per_splat.values())).shape[0]
    pix, spl = _dump_sample(H * W, DUMP_PIXELS, 1), _dump_sample(P, DUMP_SPLATS, 2)
    arrays = {}
    for k, v in images.items():
        arrays[k] = np.asarray(v, np.float32) if pix is None else np.asarray(v, np.float32).reshape(v.shape[0], -1)[:, pix]
    for k, v in per_splat.items():
        arrays[k] = np.asarray(v, np.float32) if spl is None else np.asarray(v, np.float32)[spl]
    if pix is not None:
        arrays["pixel_index"] = pix.astype(np.float64)
    if spl is not None:
        arrays["splat_index"] = spl.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"{total} bytes of outputs to dump"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))
    return sorted(arrays)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region; every sample is stamped on receipt so that only
    samples inside [mark_start, mark_stop] are reported.  Source: NVML in-process (nvidia_ml_py: the same counters
    nvidia-smi prints — SM clock and the event-reason bit mask only, two cheap calls every 10 ms, no power / SMBus reads); fallback: the profiling recipe's `nvidia-smi --query-gpu
    ... -lms 200` child process.  Round 2 measured what the sampler itself costs: `nvidia-smi -lms 20` (round 1's
    setting) stalled kernel launches for 2-13 ms a few times per 100 steps — 561 / 603 / 621 Msplats/s in three
    back-to-back runs against 624 without any sampler (profiles/r2_bench_repeat_*.json)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t0, self.t1 = index, None, [], None, None
        self.mode, self._stop = None, False

    def start(self):
        want = os.environ.get("SURFEL_BENCH_CLOCKS", "nvml")
        if want == "nvml":
            try:
                import pynvml
                pynvml.nvmlInit()
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
                self.nv = pynvml
                self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
                self.mode = "nvml"
                self.t = threading.Thread(target=self._poll_nvml, daemon=True)
                self.t.start()
                return
            except Exception:
                self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.mode = "nvidia-smi -lms 200"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t_end = time.time() + 3.0
            while not self.lines and time.time() < t_end:     # wait for the first sample
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = int(get_reasons(self.h))
                flags = ",".join("Active" if r & bits[n] else "Not Active" for n in self.NAMES)
                self.lines.append((time.time(), f"{sm}, {self.mx}, 0, {flags}"))
            except Exception:
                pass
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark_start(self):
        self.t0 = time.time()

    def mark_stop(self):
        self.t1 = time.time()

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock sampler (NVML and nvidia-smi unavailable, or SURFEL_BENCH_NOCLOCKS)"]}
        time.sleep(0.06)
        self._stop = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        names = self.NAMES

        def parse(lines):
            sm, mx, reasons = [], [], set()
            for _, ln in lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except ValueError:
                    continue
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            return sorted(sm), mx, reasons
        inside = [x for x in self.lines if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or 1e30) + 0.02]
        note = "samples inside the timed region"
        if len(inside) < 2:       # region shorter than the sampling period: widen to +-0.3 s around it
            inside = [x for x in self.lines if self.t0 is not None and self.t0 - 0.3 <= x[0] <= (self.t1 or 1e30) + 0.3]
            note = "timed region shorter than 2 sampling periods: samples within +-0.3 s of it (GPU busy with the same loop)"
        sm, mx, reasons = parse(inside)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "note": note, "source": self.mode}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs of the NUMA node the GPU hangs off, BEFORE any pinned host memory is
    allocated, so that the e2e leg's H2D/D2H copies do not cross the socket interconnect.  Best effort:
    returns the node id or None."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        if bus.startswith("00000000:"):
            bus = bus[4:]                                    # sysfs uses a 4-digit PCI domain
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def set_pinned_policy(policy):
    """Placement of the pinned host buffers of the e2e leg: "local" = on the NUMA node of the rank's GPU (CPU
    affinity + first touch, bind_to_gpu_numa_node), "interleave" = pages interleaved over all nodes
    (set_mempolicy(MPOL_INTERLEAVE) before the allocations).  Which one is faster when several ranks share a
    socket is a property of the box: profiles/pcie_concurrent.py measures both."""
    if policy != "interleave":
        return False
    try:
        import ctypes
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        mask = ctypes.c_ulong(sum(1 << n for n in nodes))
        return ctypes.CDLL(None, use_errno=True).syscall(238, ctypes.c_int(3), ctypes.byref(mask), ctypes.c_ulong(64)) == 0
    except Exception:
        return False


def cpu_oracle_run(scene_np, cam_np, gc, go, P, max_seconds=25.0):
    """C-oracle (OpenMP, all host cores) fwd+bwd.  Full workload if it fits the time budget, else a
    bounded sample: a band of tile rows of the same frame (all P splats are still preprocessed)."""
    import numpy as np
    from oracle import surfel_oracle as O
    O.build()
    O.set_threads(0)          # every host core, whatever OMP_NUM_THREADS says (torchrun exports 1 into each rank)
    bg = np.zeros(3, np.float32)
    gy = (cam_np["H"] + 15) // 16
    # probe with a thin band to estimate the cost of the full frame
    probe_rows = max(1, gy // 16)
    r0 = (gy - probe_rows) // 2
    t0 = time.perf_counter()
    pre, binned, img = O.forward(scene_np, cam_np, bg, row0=r0, row1=r0 + probe_rows)
    O.backward(scene_np, cam_np, bg, pre, binned, img, gc, go)
    t_probe = time.perf_counter() - t0
    est_full = t_probe * gy / probe_rows
    if est_full <= max_seconds:
        rows, r0 = gy, 0
    else:
        rows = max(probe_rows, int(gy * max_seconds / est_full))
        r0 = (gy - rows) // 2
    t0 = time.perf_counter()
    pre, binned, img = O.forward(scene_np, cam_np, bg, row0=r0, row1=r0 + rows)
    O.backward(scene_np, cam_np, bg, pre, binned, img, gc, go)
    dt = time.perf_counter() - t0
    frac = rows / gy
    sample = (f"full frame, {P} splats" if rows == gy else
              f"tile rows [{r0},{r0 + rows}) of {gy} ({frac:.3f} of the frame; all {P} splats preprocessed); "
              f"value = P*fraction/t")
    return P * frac / dt / 1e6, dt, sample


def run_reference(args, rank, world):
    """Reference arm: CPU restatement of the reference rasterizer on the host cores."""
    if rank != 0:
        return
    import numpy as np
    import surfel_scenes as S
    P, W, H = S.CONFIGS[args.workload]
    scene, cam = S.named(args.workload)
    gc, go = S.make_cotangents(W, H, S.CONFIG_SEED[args.workload])
    sn, cn = S.to_numpy(scene), S.to_numpy(cam)
    try:
        os.sched_setaffinity(0, range(os.cpu_count()))    # a launcher may have pinned the rank to a few cores
    except Exception:
        pass
    from oracle import surfel_oracle as O
    O.build()
    cores = O.set_threads(0)
    # CPU steps are seconds long: run at most 6 timed + 1 warm-up sample however large K is, each
    # bounded so that the whole arm ends within a few minutes; the JSON line reports the real counts.
    n_warm, n_steps = min(args.warmup, 1), min(args.steps, 6)
    per_step = max(2.0, min(25.0, 150.0 / max(1, n_steps + n_warm)))
    vals, sample = [], ""
    args.warmup, args.steps = n_warm, n_steps
    for i in range(args.warmup + args.steps):
        v, dt, sample = cpu_oracle_run(sn, cn, gc.numpy(), go.numpy(), P, max_seconds=per_step)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.workload, P, W, H),
                   "note": "one host serves every view: at N GPUs the repo arm renders N views per step on N devices, this arm is "
                           "the throughput of the box's host cores on the same per-view workload"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference CUDA rasterizer is not vendored in /root/reference; this is the CPU restatement (oracle/)",
    }
    _emit(json.dumps(out))


def tile_band_leg(rank, world, dev, steps=6, warmup=2, workload="config5"):
    """Second leg at N > 1 (SURVEY §8e, BASELINE config 5): ONE oversized frame rendered in N tile-row bands,
    the band outputs completed by in-place all-gathers over NVLink, the per-splat gradients summed by one
    all-reduce of the op's flat gradient bucket.  Device times (CUDA events), max over ranks."""
    import torch
    import torch.distributed as dist
    import surfel_parallel as SP
    import surfel_scenes as S
    from diff_surfel_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    P, W, H = S.CONFIGS[workload]
    scene, cam = S.named(workload)                       # same seed on every rank: replicated splats
    rs = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"], bg=torch.zeros(3, device=dev),
        scale_modifier=1.0, viewmatrix=cam["viewmatrix"].to(dev), projmatrix=cam["projmatrix"].to(dev), sh_degree=3,
        campos=cam["campos"].to(dev), prefiltered=False, debug=False)
    names = ("means3D", "scales", "rotations", "opacities", "shs")
    leaf = {k: scene[k].to(dev).requires_grad_(True) for k in names}
    m2d = torch.zeros(P, 3, device=dev, requires_grad=True)
    gc, go = S.make_cotangents(W, H, 5)
    gc, go = gc.to(dev), go.to(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
    acc = [0.0] * 6

    def step(timed):
        for t in list(leaf.values()) + [m2d]:
            t.grad = None
        ev[0].record()
        res = SP.rasterize_tile_band(GaussianRasterizer, rs, rank, world, grad_reduce="defer", means3D=leaf["means3D"],
                                     means2D=m2d, shs=leaf["shs"], opacities=leaf["opacities"], scales=leaf["scales"],
                                     rotations=leaf["rotations"])
        ev[1].record()                                                       # band forward + in-place all-gathers
        torch.autograd.backward([res["render"], res["allmap"]], [gc, go])    # cotangents read in place, band backward
        ev[2].record()
        frame, bucket = SP.last_exchange_buffers()
        dist.all_reduce(bucket)                                              # sum of the band partials (16 floats per splat), one collective
        if SP.last_sh_expand() is not None:
            SP.last_sh_expand()()                                            # SH gradient = basis (x) summed colour gradient
        ev[3].record()
        # the collectives once more on the same buffers, alone (the gather is idempotent; the second all-reduce
        # only scales this step's throw-away gradients), so that their cost can be separated from the kernels'
        ev[4].record()
        SP.allgather_frame_inplace(frame, H, rank, world)
        ev[5].record()
        shard = torch.empty(bucket.numel() // world, device=dev) if bucket.numel() % world == 0 else None
        if shard is not None:
            dist.reduce_scatter_tensor(shard, bucket)
        ev[6].record()
        torch.cuda.synchronize()
        if timed:
            for i, (a, b) in enumerate(((0, 1), (1, 2), (2, 3), (4, 5), (5, 6), (0, 3))):
                acc[i] += ev[a].elapsed_time(ev[b])
        return res

    shard_buf = {}

    def reduce_grads(bucket, reduce):
        if reduce == "all_reduce":
            dist.all_reduce(bucket)
        else:
            if "t" not in shard_buf:
                shard_buf["t"] = torch.empty(bucket.numel() // world, device=dev)
            dist.reduce_scatter_tensor(shard_buf["t"], bucket)
        if SP.last_sh_expand() is not None:
            SP.last_sh_expand()()

    def step_variant(gather, reduce, acc_key):
        """The same frame with the exchange taken off the critical path.
        gather="async": the all-gathers are only enqueued and the band backward (which reads this band's cotangent
        rows only) runs while they are in flight — what a band-local loss permits.
        gather="fused"/"fused_p2p": no all-gather at all; the render kernel stores the band into every GPU's copy of
        the frame (NVSwitch multicast / peer stores over NVLink) and a cross-GPU barrier follows.
        Either way the full frame is complete, and the gradients reduced, at the end of the timed region."""
        for t in list(leaf.values()) + [m2d]:
            t.grad = None
        ev[0].record()
        res = SP.rasterize_tile_band(GaussianRasterizer, rs, rank, world, grad_reduce="defer", gather=gather,
                                     means3D=leaf["means3D"], means2D=m2d, shs=leaf["shs"], opacities=leaf["opacities"],
                                     scales=leaf["scales"], rotations=leaf["rotations"])
        ev[1].record()
        torch.autograd.backward([res["render"], res["allmap"]], [gc, go])
        _, bucket = SP.last_exchange_buffers()
        reduce_grads(bucket, reduce)
        res["wait"]()                                                        # the frame is complete on this stream
        ev[2].record()
        torch.cuda.synchronize()
        acc_var[acc_key] = acc_var.get(acc_key, 0.0) + ev[0].elapsed_time(ev[2])
        acc_var[acc_key + ":fwd"] = acc_var.get(acc_key + ":fwd", 0.0) + ev[0].elapsed_time(ev[1])
        return res

    acc_var = {}

    import ctypes
    import time as _time
    from diff_surfel_rasterization import _cabi
    lib = _cabi.load()
    for _ in range(warmup):
        res = step(False)
    dist.barrier(); torch.cuda.synchronize()
    nst = lib.surfel_profile_num_stages()
    ms_arr, cnt_arr = (ctypes.c_double * nst)(), (ctypes.c_int * nst)()
    lib.surfel_profile_enable(1); lib.surfel_profile_read(ms_arr, cnt_arr)
    t_host = _time.perf_counter()
    for _ in range(steps):
        res = step(True)
    t_host = (_time.perf_counter() - t_host) / steps * 1e3
    lib.surfel_profile_enable(0); lib.surfel_profile_read(ms_arr, cnt_arr)
    kernels = {lib.surfel_profile_stage_name(i).decode(): round(ms_arr[i] / steps, 3) for i in range(nst) if cnt_arr[i]}
    # (gather="async" — NCCL gathers hidden behind the backward — was measured and dropped from the default run:
    # 9.2 vs 8.9 ms at N = 2, 10.7 vs 5.6 ms at N = 8; profiles/r2_bench_8gpu_a.json)
    variants = [("fused", "all_reduce", "fused"), ("fused_multicast", "all_reduce", "fused_multicast")]
    var_ms, var_err, var_res, fused_via = {}, {}, {}, {}
    for gather, reduce, key in variants:
        try:
            step_variant(gather, reduce, key)                                # one untimed step per variant
            acc_var.pop(key, None); acc_var.pop(key + ":fwd", None)
            dist.barrier(); torch.cuda.synchronize()
            for _ in range(steps):
                var_res[key] = step_variant(gather, reduce, key)
            fused_via[key] = SP._last.get("fused_via") if gather.startswith("fused") else None
            tv = torch.tensor([acc_var[key] / steps, acc_var[key + ":fwd"] / steps], device=dev, dtype=torch.float64)
            dist.all_reduce(tv, op=dist.ReduceOp.MAX)
            var_ms[key] = (float(tv[0]), float(tv[1]))
        except Exception as ex:     # noqa: BLE001 — e.g. no symmetric memory / multicast on this box: reported, not hidden
            var_err[key] = f"{type(ex).__name__}: {ex}"[:300]
    tt = torch.tensor([a / steps for a in acc], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    fwd_total, bwd, allreduce, gather, rscatter, frame = (float(x) for x in tt)
    out = {"workload": f"{workload}: {P} surfels, one {W}x{H} frame in {world} tile-row bands",
           "ms_frame": frame, "ms_band_fwd": max(0.0, fwd_total - gather), "ms_allgather": gather, "ms_band_bwd": bwd,
           "ms_allreduce": allreduce, "ms_reduce_scatter_alternative": rscatter,
           "gather_bytes_per_rank": int(10 * 4 * W * SP.equal_band_rows(H, world) * 16),
           "grad_bytes": int(SP.last_exchange_buffers()[1].numel() * 4),
           "ms_frame_overlapped": var_ms.get("overlapped", (None,))[0],
           "overlapped": "all-gathers enqueued asynchronously and hidden behind the band backward (band-local cotangents), "
                         "then the gradient all-reduce / reduce-scatter; full frame complete at the end of the step",
           "ms_frame_fused": var_ms.get("fused", (None,))[0], "ms_band_fwd_fused": var_ms.get("fused", (None, None))[1],
           "ms_frame_fused_reduce_scatter": var_ms.get("fused_rs", (None,))[0],
           "ms_frame_fused_multicast": var_ms.get("fused_multicast", (None,))[0],
           "ms_band_fwd_fused_multicast": var_ms.get("fused_multicast", (None, None))[1],
           "fused": "no all-gather: the render kernel stores its band into every GPU's copy of the frame in symmetric "
                    "memory over NVLink (one store per peer and value; fused_multicast = one store per value to the "
                    "NVSwitch multicast address), then a cross-GPU barrier; ms_band_fwd_fused = band forward + exchange + "
                    "barrier, to compare with ms_band_fwd + ms_allgather",
           "variant_errors": var_err or None,
           "Msplats_per_s": P / frame / 1e3, "steps": steps, "kernel_ms_rank0": kernels, "host_ms_per_step_rank0": t_host,
           "how": "padded frame, bands rendered in place, one in-place all_gather_into_tensor per plane; cotangents read in "
                  "place; one all_reduce of the flat gradient bucket — 16 floats per splat: the SH gradient is expanded from "
                  "the summed colour gradient after the reduction (ms_allreduce includes that expansion; reduce-scatter "
                  "timed as the sharded-optimizer alternative)"}
    cands = {"nccl in-place all-gather + all-reduce": frame}
    for key, label in (("overlapped", "asynchronous all-gather + all-reduce"), ("fused", "exchange fused into the render kernel + all-reduce"),
                       ("fused_multicast", "fused via NVSwitch multicast + all-reduce"),
                       ("fused_rs", "exchange fused into the render kernel + reduce-scatter (sharded optimizer)")):
        if key in var_ms:
            cands[label] = var_ms[key][0]
    best = min(cands, key=cands.get)
    out["best"] = {"variant": best, "ms_frame": cands[best], "Msplats_per_s": P / cands[best] / 1e3}
    if rank == 0:
        # the completed frame against ONE GPU rendering the whole frame
        with torch.no_grad():
            color, radii, allmap = GaussianRasterizer(rs)(means3D=leaf["means3D"], means2D=m2d, shs=leaf["shs"],
                                                          opacities=leaf["opacities"], scales=leaf["scales"], rotations=leaf["rotations"])
        out["stitched_equals_single_gpu"] = bool(torch.equal(res["render"], color) and torch.equal(res["allmap"], allmap)
                                                 and torch.equal(res["radii"], radii)
                                                 and all(torch.equal(r["render"], color) and torch.equal(r["allmap"], allmap)
                                                         for r in var_res.values()))
        out["variants_checked"] = sorted(var_res)
    dist.barrier()
    return out


def run_ours(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    import surfel_scenes as S
    import diff_surfel_rasterization as dsr
    from diff_surfel_rasterization import GaussianRasterizationSettings, GaussianRasterizer, _cabi

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    numa_node = None if os.environ.get("SURFEL_BENCH_NO_NUMA") else bind_to_gpu_numa_node(local_rank)
    pin_interleaved = set_pinned_policy(args.pin_policy)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _cabi.load()
    P, W, H = S.CONFIGS[args.workload]
    if args.splats:
        P = args.splats
    cam = S.make_camera(W, H)
    # independent views: every rank renders its own statistically identical scene/view
    scene = S.make_scene(P, W, H, S.CONFIG_SEED[args.workload] + 1000 * rank)
    gc_h, go_h = S.make_cotangents(W, H, S.CONFIG_SEED[args.workload] + rank)
    names = ["means3D", "scales", "rotations", "opacities", "shs"]
    host_in = {k: scene[k].pin_memory() for k in names}
    host_gc, host_go = gc_h.pin_memory(), go_h.pin_memory()
    bg = torch.zeros(3, device=dev)
    rs = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"], bg=bg, scale_modifier=1.0,
        viewmatrix=cam["viewmatrix"].to(dev), projmatrix=cam["projmatrix"].to(dev), sh_degree=3,
        campos=cam["campos"].to(dev), prefiltered=False, debug=False)
    rast = GaussianRasterizer(rs)
    leaf = {k: host_in[k].to(dev).requires_grad_(True) for k in names}
    means2D = torch.zeros(P, 3, device=dev, requires_grad=True)
    gc, go = host_gc.to(dev), host_go.to(dev)

    def step(inp, m2d, gcd, god):
        for t in list(inp.values()) + [m2d]:
            t.grad = None
        color, radii, allmap = rast(means3D=inp["means3D"], means2D=m2d, shs=inp["shs"], opacities=inp["opacities"],
                                    scales=inp["scales"], rotations=inp["rotations"])
        torch.autograd.backward([color, allmap], [gcd, god])
        return color, radii, allmap

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput ("value") ----
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("SURFEL_BENCH_NOCLOCKS"):
        sampler.start()
    for _ in range(args.warmup):
        color, radii, allmap = step(leaf, means2D, gc, go)
    torch.cuda.synchronize()
    V = int((radii > 0).sum())
    R = int(dsr.last_num_rendered())
    barrier()
    n_stage = lib.surfel_profile_num_stages()
    import ctypes
    ms_arr, cnt_arr = (ctypes.c_double * n_stage)(), (ctypes.c_int * n_stage)()
    launches0 = lib.surfel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Python's cyclic garbage collector is paused inside the timed regions (collected right before): a
    # generation-2 pass over the heap of a process with torch and a 1 M-splat scene loaded takes milliseconds, i.e.
    # several steps' worth of a 20-step window on whichever rank it hits.  A precaution — the host stalls actually
    # seen in round 2 came from the nvidia-smi clock sampler (see ClockSampler).  The op itself creates no
    # reference cycles (tests/test_parity_gpu.py::test_out_buffers_are_not_kept_alive_by_the_graph runs with the
    # collector off), so nothing accumulates.
    import gc as _gc
    pause_gc = not os.environ.get("SURFEL_BENCH_KEEP_GC")
    if pause_gc:
        _gc.collect()
        _gc.disable()
    sampler.mark_start()
    host_ts = [time.perf_counter()]          # diagnostic only: when the host finished issuing each step
    e0.record()
    for _ in range(args.steps):
        last = None           # free the previous step's outputs first: the allocator reuses their blocks, as without --dump-outputs
        last = step(leaf, means2D, gc, go)
        host_ts.append(time.perf_counter())
    e1.record()
    torch.cuda.synchronize()
    sampler.mark_stop()
    _gc.enable()
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the passes below overwrite the gradients
        out_color, out_radii, out_allmap = last
        grads = {f"grad_{k}": leaf[k].grad for k in names}
        grads["grad_means2D"] = means2D.grad
        dump_outputs(args.dump_outputs, {"color": out_color.detach().cpu().numpy(), "allmap": out_allmap.detach().cpu().numpy()},
                     {"radii": out_radii.cpu().numpy(), **{k: g.cpu().numpy() for k, g in grads.items()}})
    del last
    launches = int(lib.surfel_launch_count() - launches0)
    # second pass, same loop, with CUDA events recorded around every kernel on the launching stream:
    # per-kernel durations for the roofline (kept out of the pass that produces `value`)
    prof_steps = max(3, min(args.steps, 50))
    lib.surfel_profile_enable(1)
    lib.surfel_profile_read(ms_arr, cnt_arr)   # drain
    for _ in range(prof_steps):
        step(leaf, means2D, gc, go)
    torch.cuda.synchronize()
    lib.surfel_profile_enable(0)
    lib.surfel_profile_read(ms_arr, cnt_arr)
    clocks = sampler.stop() if rank == 0 else None
    t_ms = e0.elapsed_time(e1)
    # per-step host intervals (the host runs at most one R-wait ahead of the device, so in steady state they
    # track the device step time; isolated long ones are host hiccups): median / p95 / max, worst rank
    iv = sorted((b - a) * 1e3 for a, b in zip(host_ts[:-1], host_ts[1:]))
    host_iv = [iv[len(iv) // 2], iv[min(len(iv) - 1, int(0.95 * len(iv)))], iv[-1]] if iv else [0.0, 0.0, 0.0]
    tt = torch.tensor([t_ms] + host_iv, device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    barrier()
    t_ms = float(tt[0].item())
    host_step_ms = {"median": float(tt[1].item()), "p95": float(tt[2].item()), "max": float(tt[3].item()),
                    "what": "host-side interval between consecutive steps of the timed loop, max over ranks (diagnostic)"}
    ms_per_step = t_ms / args.steps
    value = world * P / (ms_per_step * 1e-3) / 1e6

    stage = {lib.surfel_profile_stage_name(i).decode(): (ms_arr[i], cnt_arr[i]) for i in range(n_stage) if cnt_arr[i]}
    per_step = {k: v[0] / prof_steps for k, v in stage.items()}            # ms per step, all launches
    per_launch = {k: v[0] / v[1] for k, v in stage.items()}                # ms per launch
    alg = algorithmic_bytes(P, V, R, W, H)
    alg_launch = dict(alg)                                                 # bytes per LAUNCH
    alg_launch["sort_onesweep_pass"] = 24 * R                              # one read + one write of the pairs
    alg_launch["sort_histogram"] = 8 * R
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    alg_launch.update({"tile_count": 20 * V + 4 * R, "tile_scan": 16 * tiles, "tile_scatter": 20 * V + 12 * R,
                       "tile_sort": 12 * R / 2})                           # two launches (small + large lists) share 12 B/instance
    peak, peak_src = measured_peak()
    dom = max(per_step, key=lambda k: per_step[k])
    achieved = alg_launch[dom] / (per_launch[dom] * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(dom)
        except Exception:
            traffic = None
    ncu_stats = None
    spath = os.path.join(ROOT, "profiles", "ncu_kernel_stats.json")
    if os.path.exists(spath):
        try:
            ncu_stats = json.load(open(spath)).get(dom)
        except Exception:
            ncu_stats = None
    b_alg = sum(alg.values())
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_launch[dom], "kernel_ms_per_launch": per_launch[dom],
                "kernel_share_of_step": per_step[dom] / ms_per_step,
                "kernel_timing": f"CUDA events around every launch, second pass of {prof_steps} steps right after the timed region",
                # the render kernels are instruction-issue bound, not HBM bound (SURVEY §8d): ncu's view of
                # the same kernel (committed capture, profiles/), reported next to the HBM fraction
                "ncu": ncu_stats,
                "pipeline": {"algorithmic_bytes": b_alg, "ms": ms_per_step,
                             "achieved": b_alg / (ms_per_step * 1e-3) / 1e9,
                             "frac": b_alg / (ms_per_step * 1e-3) / 1e9 / peak},
                "stage_ms_per_step": {k: round(v, 4) for k, v in per_step.items()},
                "stage_frac_of_peak": {k: round(alg_launch[k] / (per_launch[k] * 1e-3) / 1e9 / peak, 4)
                                       for k in per_launch if k in alg_launch}}

    # ---- end to end with HOST buffers (H2D of every input, D2H of outputs + gradients) ----
    host_out = {"color": torch.empty(3, H, W).pin_memory(), "allmap": torch.empty(7, H, W).pin_memory(),
                "radii": torch.empty(P, dtype=torch.int32).pin_memory()}
    host_grad = {k: torch.empty_like(scene[k]).pin_memory() for k in names}
    host_grad["means2D"] = torch.empty(P, 3).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in host_in.values()) + host_gc.numel() * 4 + host_go.numel() * 4
    d2h = sum(t.numel() * t.element_size() for t in list(host_out.values()) + list(host_grad.values()))

    e2e = None
    if not args.no_e2e:
        # the repo's public host-buffer API: three-stream software pipeline (surfel_host.py); every
        # step still moves all of its inputs H2D and all of its results D2H inside the timed region
        from surfel_host import HostStepPipeline
        pipe = HostStepPipeline(rast, host_in, host_gc, host_go, dev)
        pipe.run(max(2, min(args.warmup, 3)), host_in, host_gc, host_go, host_out, host_grad)
        barrier()
        e2e_steps = max(4, min(args.steps, 50))     # >= 4 so that the 3-stage pipeline reaches steady state
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if pause_gc and not os.environ.get("SURFEL_BENCH_E2E_KEEP_GC"):
            _gc.collect(); _gc.disable()
        ea.record(pipe.s_in)
        pipe.run(e2e_steps, host_in, host_gc, host_go, host_out, host_grad)
        eb.record(pipe.s_out)
        torch.cuda.synchronize()
        _gc.enable()
        te = torch.tensor([ea.elapsed_time(eb)], device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        barrier()
        e2e_ms = float(te.item()) / e2e_steps
        # sanity: the host buffers really hold this step's results
        # the host buffers must hold THIS workload's results: the forward is bit-deterministic, so color / allmap /
        # radii that came back over PCIe equal the resident run's exactly; gradients agree up to atomic ordering
        ref_c, ref_r, ref_a = step(leaf, means2D, gc, go)
        torch.cuda.synchronize()
        def _close(a, b):
            return float((a - b).abs().max()) <= 1e-4 * float(b.abs().max()) + 1e-30
        ok = bool(torch.equal(host_out["color"], ref_c.detach().cpu()) and torch.equal(host_out["allmap"], ref_a.detach().cpu())
                  and torch.equal(host_out["radii"], ref_r.cpu())
                  and all(_close(host_grad[k], leaf[k].grad.cpu()) for k in names)
                  and _close(host_grad["means2D"], means2D.grad.cpu()))
        e2e = {"value": world * P / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": e2e_ms, "steps": e2e_steps,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "results_checked": ok,
               "results_check": "host copies of color / allmap / radii bit-equal to the resident run, gradients within 1e-4 of their max",
               "how": "pinned host buffers; H2D / compute / D2H pipelined on 3 streams (surfel_host.HostStepPipeline)"}

    # ---- CPU baseline on rank 0 (N == 1 only) ----
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            os.sched_setaffinity(0, range(os.cpu_count()))   # the CPU leg uses every host core again
        except Exception:
            pass
        sn, cn = S.to_numpy(scene), S.to_numpy(cam)
        v, dt, sample = cpu_oracle_run(sn, cn, gc_h.numpy(), go_h.numpy(), P, max_seconds=20.0)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                        "sample": sample, "seconds": dt}
        try:   # the "pure-Python surfel rasterizer" of BASELINE.md §2.1 (dense PyTorch, config 1, forward)
            from oracle import dense_torch as DT
            s1, c1 = S.named("config1")
            torch.set_num_threads(min(32, os.cpu_count()))
            ts = []
            for _ in range(1):
                t0 = time.perf_counter()
                with torch.no_grad():
                    DT.render(s1["means3D"], s1["scales"], s1["rotations"], s1["opacities"], s1["shs"], c1["viewmatrix"],
                              c1["projmatrix"], c1["campos"], torch.zeros(3), c1["W"], c1["H"], pixel_chunk=8192)
                ts.append(time.perf_counter() - t0)
            cpu_baseline["pure_python_config1_forward"] = {"ms": sorted(ts)[0] * 1e3, "Msplats_per_s": 1000 / sorted(ts)[0] / 1e6,
                                                           "what": "dense PyTorch surfel rasterizer, 1k surfels 256x256, forward only"}
        except Exception as ex:   # never let the optional extra break the bench line
            cpu_baseline["pure_python_config1_forward"] = {"error": str(ex)[:200]}

    # ---- tile-band leg (N > 1): ONE config-5 frame in N bands, exchange over NVLink ----
    tile_band = None
    if world > 1 and not args.no_tile_band:
        try:
            del leaf, means2D, gc, go
            torch.cuda.empty_cache()
            tile_band = tile_band_leg(rank, world, dev)
        except Exception as ex:      # the headline line must survive a failure of the second leg
            tile_band = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.workload, P, W, H),
                       "visible": V, "instances": R, "parallelism": f"view-parallel x{world} (no collective)",
                       "host_numa_node": numa_node, "pinned_buffers": "interleaved over NUMA nodes" if pin_interleaved else "local to the GPU's NUMA node",
                       "l2_policy": "inputs larger than L2 (232 MB of splat parameters + 83 MB of outputs per step vs 126 MB L2)",
                       "host_gc": "python cyclic garbage collector paused inside the timed regions (collected right before)"},
            "e2e": e2e, "gpu_launches": launches, "gpu_launches_per_step": launches / args.steps,
            "roofline": roofline, "clocks": clocks, "host_step_ms": host_step_ms,
        }
        if cpu_baseline is not None:
            out["cpu_baseline"] = cpu_baseline
        if tile_band is not None:
            out["tile_band"] = tile_band
        _emit(json.dumps(out))


class _CleanStdout:
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its
    version banner when NCCL_DEBUG is set, OpenMP runtimes warn, ...), so for the duration of the run file
    descriptor 1 points at stderr and the JSON line is written to the saved, real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.real, (line.rstrip("\n") + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.real, 1)
        os.close(self.real)
        return False


_emit = print          # replaced by _CleanStdout.emit while main() runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="headline")
    ap.add_argument("--splats", type=int, default=0, help="override P (debugging only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs only)")
    ap.add_argument("--pin-policy", choices=["local", "interleave"], default=os.environ.get("SURFEL_PIN_POLICY", "local"),
                    help="NUMA placement of the e2e leg's pinned host buffers")
    ap.add_argument("--no-tile-band", action="store_true", help="skip the tile-band leg that runs at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs and gradients (rank 0) as DIR/<name>.npy, at most 64 MB: "
                         "a fixed, seeded sample of pixels and splats at large sizes")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the timed path of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    global _emit
    with _CleanStdout() as out:
        _emit = out.emit
        try:
            if args.impl == "reference":
                run_reference(args, rank, world)
                return
            if world > 1:
                import torch
                import torch.distributed as dist
                torch.cuda.set_device(local_rank)
                dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            try:
                run_ours(args, rank, local_rank, world)
            finally:
                if world > 1:
                    import torch.distributed as dist
                    dist.destroy_process_group()
        finally:
            _emit = print


if __name__ == "__main__":
    main()
