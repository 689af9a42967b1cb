#!/usr/bin/env python
"""bench.py -- images/s of the ctdet heat-map decode hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one ctdet_decode pass (3x3 peak-NMS + top-K + wh/reg gather + box assembly)
over one synthetic batch: BASELINE configs[1] geometry, 64 images per GPU of
80x128x128 post-sigmoid heat + wh + reg, K=100.  Weak scaling: every rank decodes its
own 64-image shard, no data-path collective (SURVEY.md section 8e).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events, max
over ranks); `e2e` = same metric through the public API with pinned HOST buffers, the
H2D of the heat/wh/reg batch and the D2H of the detections inside the timed region;
`roofline` = algorithmic bytes / device time against MEASURED_PEAKS.json;
`cpu_baseline` = the CPU port of the reference path on a bounded sample.

--dump-outputs DIR writes the detections of the last timed step, [64, K, 6] float32, to DIR/dets.npy
(DIR/dets.rank<r>.npy per rank when N > 1).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "images/sec ctdet 512x512->128x128x80 heatmap decode K=100"
UNIT = "images/s"
B_PER_GPU, C, H, W, K = 64, 80, 128, 128, 100
ALG_BYTES_PER_IMAGE = C * H * W * 4 + K * 4 * 4 + K * 6 * 4   # SURVEY.md section 8d: 5,246,880 B
N_ROT = 3                                                      # rotating input batches (3 x 352 MB >> 126 MB L2)
NCU_TRAFFIC_BYTES = 341761536 + 3631360                        # measured DRAM read + write of one launch (profiles/r2)


def workload_config(world):
    """The SAME dict in both arms (the driver compares them): what one step processes."""
    return {
        "workload": "ctdet decode, %d img/GPU x %dx%dx%d post-sigmoid heat + wh + reg, K=%d "
                    "(BASELINE configs[1] geometry: DLA-34 512x512 batch=64 heads)" % (B_PER_GPU, C, H, W, K),
        "global_batch": B_PER_GPU * world,
        "parallelism": "dp%d (batch shards, no collective)" % world,
        "l2": "inputs > L2: %d rotating batches of %.0f MB" % (N_ROT, B_PER_GPU * (C + 4) * H * W * 4 / 1e6),
    }


def _nvml_handle(cuda_index):
    """NVML handle of CUDA device `cuda_index`.  NVML enumerates every GPU of the box while CUDA sees only the
    visible ones (CUDA_VISIBLE_DEVICES), so the two indices differ: match through the PCI bus id."""
    import pynvml as nv
    nv.nvmlInit()
    p = torch.cuda.get_device_properties(cuda_index)
    if all(hasattr(p, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
        bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        try:
            return nv, nv.nvmlDeviceGetHandleByPciBusId(bus.encode()), bus
        except Exception:
            pass
    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    ids = [v.strip() for v in vis.split(",") if v.strip()]
    if cuda_index < len(ids):
        v = ids[cuda_index]
        try:
            h = nv.nvmlDeviceGetHandleByUUID(v.encode()) if v.startswith("GPU-") else nv.nvmlDeviceGetHandleByIndex(int(v))
            return nv, h, "visible:" + v
        except Exception:
            pass
    return nv, nv.nvmlDeviceGetHandleByIndex(cuda_index), "index:%d" % cuda_index


def bind_to_gpu_numa_node(index):
    """Pin this rank (and the pinned host buffers it allocates afterwards, first touch) to the NUMA node its
    GPU hangs off: at N=8 the eight H2D streams otherwise fight over one socket's memory controllers.
    Returns a short description for the JSON line."""
    try:
        nv, h, how = _nvml_handle(index)
        bus = nv.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/numa_node" % (dom[-4:].lower(), rest.lower())
        node = int(open(path).read().strip())
        if node < 0:
            return "numa_node unknown (single node), gpu %s" % bus
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "not bound (node %d has no allowed cpu), gpu %s" % (node, bus)
        os.sched_setaffinity(0, allowed)
        return "gpu %s (%s) -> NUMA node %d, %d cpus" % (bus, how, node, len(allowed))
    except Exception as e:
        return "not bound (%s)" % type(e).__name__


def synth(batch, device, seed):
    """SURVEY.md section 8d synthetic inputs: heat = sigmoid(randn - 2.19), wh = rand*32, reg = rand."""
    g = torch.Generator(device=device).manual_seed(seed)
    heat = torch.sigmoid(torch.randn(batch, C, H, W, device=device, generator=g) - 2.19)
    wh = torch.rand(batch, 2, H, W, device=device, generator=g) * 32
    reg = torch.rand(batch, 2, H, W, device=device, generator=g)
    return heat, wh, reg


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.recording = False      # only samples taken inside the timed region are kept ...
        self.sample_now = False     # ... plus one forced sample right before it (GPU under warm-up load) and after it
        self.alive = threading.Event()

    def run(self):
        try:
            nv, h, _ = _nvml_handle(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            while not self.stop_flag:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.alive.set()
                if self.recording or self.sample_now:
                    self.sample_now = False
                    self.samples.append(mhz)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                if not self.recording:
                    time.sleep(0.0005)          # back-to-back NVML reads (~50 us each) inside the timed region
        except Exception as e:  # no NVML: report that instead of inventing numbers
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)
            self.alive.set()

    def force_sample(self):
        """One synchronous sample (the driver's 20-step region lasts < 2 ms, shorter than a scheduling quantum)."""
        self.sample_now = True
        t0 = time.perf_counter()
        while self.sample_now and time.perf_counter() - t0 < 0.05 and self.is_alive():
            time.sleep(0.0002)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_port_rate(batch, repeats, threads):
    """images/s of the CPU port of the reference path (oracle/torch_port.py) on `batch` images."""
    from oracle import torch_port
    torch.set_num_threads(threads)
    heat, wh, reg = synth(batch, "cpu", 317)
    torch_port.ctdet_decode(heat, wh, reg, K=K)  # warm-up
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        torch_port.ctdet_decode(heat, wh, reg, K=K)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return batch / ts[len(ts) // 2], ts


def _calibrate_cpu(cores):
    """Pick the faster of {all host threads, 8 threads} for the CPU port and return (threads, s/image)."""
    from oracle import torch_port
    heat, wh, reg = synth(4, "cpu", 317)
    best = None
    for th in sorted({cores, min(cores, 8)}, reverse=True):
        torch.set_num_threads(th)
        torch_port.ctdet_decode(heat, wh, reg, K=K)
        t0 = time.perf_counter()
        torch_port.ctdet_decode(heat, wh, reg, K=K)
        dt = (time.perf_counter() - t0) / 4
        if best is None or dt < best[1]:
            best = (th, dt)
    torch.set_num_threads(best[0])
    return best


def run_reference(args, rank, world):
    """Reference arm: the CPU port of the reference's PyTorch path on the host cores (rank 0 only).
    Each step decodes a bounded sample of the 64-image batch, sized so the run ends in ~2 minutes."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    from oracle import torch_port
    threads, s_per_img = _calibrate_cpu(cores)
    budget_s = 100.0
    sample_b = int(max(1, min(B_PER_GPU, budget_s / max(args.steps + args.warmup, 1) / s_per_img)))
    heat, wh, reg = synth(sample_b, "cpu", 317)
    for _ in range(args.warmup):
        torch_port.ctdet_decode(heat, wh, reg, K=K)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        torch_port.ctdet_decode(heat, wh, reg, K=K)
    dt = time.perf_counter() - t0
    value = sample_b * args.steps / dt
    sample = ("each step = %d of the %d images of a batch (same synthetic distribution), torch CPU op port "
              "(oracle/torch_port.py), %d threads" % (sample_b, B_PER_GPU, threads))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bind-numa", dest="bind_numa", action="store_true", default=None,
                    help="pin the rank to its GPU's NUMA node before allocating (default: only when world > 1)")
    ap.add_argument("--no-bind-numa", dest="bind_numa", action="store_false")
    ap.add_argument("--no-secondary", action="store_true", help="skip the per-kernel secondary measurements (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detections of the last timed step to DIR/dets.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm decodes a host-timed sample of the batch whose size varies from run to run
        ap.error("--dump-outputs needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the decode path has no CPU fallback")
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Host placement of the e2e leg.  (Earlier r2 runs that bound a single rank measured 11-16 GB/s: that was the
    # OpenMP team of the host process spinning on the 64 bound cores, fixed since by the single intra-op thread.)
    # N > 1: every rank keeps its pinned staging buffers on its own GPU's NUMA node (the 8-rank runs measured 43-53 GB/s
    # per rank unbound, run to run, and 52.3 GB/s bound); N = 1: the default placement measured fastest
    bind = args.bind_numa if args.bind_numa is not None else world > 1
    numa = bind_to_gpu_numa_node(local) if bind else "not bound (--bind-numa to bind)"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import centernet_b200
    from centernet_b200 import decode as D
    from centernet_b200._lib import C as CL

    batches = [synth(B_PER_GPU, dev, 317 + 1000 * rank + i) for i in range(N_ROT)]
    for i in range(max(args.warmup, 3)):
        D.ctdet_decode(*batches[i % N_ROT][:2], reg=batches[i % N_ROT][2], K=K)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (CUDA events on the launching stream)
    sampler = ClockSampler(local)
    sampler.start()
    sampler.alive.wait(timeout=10)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(3):                      # keep the GPU under load while the "before" sample is taken
        D.ctdet_decode(*batches[i % N_ROT][:2], reg=batches[i % N_ROT][2], K=K)
    sampler.force_sample()
    barrier()
    l0 = CL.launch_count()
    sampler.recording = True
    ev0.record()
    for i in range(args.steps):
        h, w_, r = batches[i % N_ROT]
        dets = D.ctdet_decode(h, w_, reg=r, K=K)
    ev1.record()
    barrier()
    sampler.recording = False
    sampler.force_sample()
    launches = CL.launch_count() - l0
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "dets.npy" if world == 1 else "dets.rank%d.npy" % rank
        np.save(os.path.join(args.dump_outputs, name), dets.float().cpu().numpy())
    sampler.stop_flag = True
    sampler.join(timeout=2)
    t = torch.tensor([ms], device=dev)
    per_rank_ms = [ms]
    if world > 1:
        allms = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(allms, t)
        per_rank_ms = [float(x.item()) for x in allms]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = B_PER_GPU * world * args.steps / (ms_max * 1e-3)

    # ---------------- secondary (SURVEY 8d): fused-sigmoid variant, input = the head's raw logits
    logit_value = None
    try:
        lg = [torch.logit(b[0].clamp(1e-7, 1 - 1e-7)) for b in batches]
        for i in range(3):
            D.ctdet_decode_from_logits(lg[i % N_ROT], batches[i % N_ROT][1], reg=batches[i % N_ROT][2], K=K)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(args.steps):
            D.ctdet_decode_from_logits(lg[i % N_ROT], batches[i % N_ROT][1], reg=batches[i % N_ROT][2], K=K)
        g1.record()
        barrier()
        tl = torch.tensor([g0.elapsed_time(g1)], device=dev)
        if world > 1:
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        logit_value = B_PER_GPU * world * args.steps / (float(tl.item()) * 1e-3)
        del lg
    except Exception as e:  # secondary number only: never take the headline down with it
        logit_value = "failed: %s" % (str(e)[:80],)

    # ---------------- end-to-end: pinned host buffers -> H2D -> decode -> D2H of the detections
    h2d = sum(x.numel() * 4 for x in batches[0])
    d2h = B_PER_GPU * K * 6 * 4
    e2e_value = None
    if args.e2e_steps > 0:
        # one intra-op thread for the host side of this leg (what torchrun sets for every rank anyway): with the
        # default of one thread per core the OpenMP team woken by the small host-side tensor ops spins on all
        # cores and the chunked copy pipeline falls to half the link rate (measured r2: 25 vs 54 GB/s)
        host_threads = torch.get_num_threads()
        torch.set_num_threads(1)
        host = [tuple(x.cpu().pin_memory() for x in batches[i]) for i in range(2)]
        # what the link gives a plain pinned copy of the same buffers right now (shared hosts vary a lot)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        batches[0][0].copy_(host[0][0], non_blocking=True)
        torch.cuda.synchronize()
        p0.record()
        for _ in range(3):
            batches[0][0].copy_(host[0][0], non_blocking=True)
        p1.record()
        torch.cuda.synchronize()
        h2d_probe = 3 * host[0][0].numel() * 4 / (p0.elapsed_time(p1) * 1e-3) / 1e9
        for i in range(2):
            D.ctdet_decode_from_host(*host[i % 2][:2], reg=host[i % 2][2], K=K)
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.e2e_steps):
            out = D.ctdet_decode_from_host(*host[i % 2][:2], reg=host[i % 2][2], K=K)   # returns a host tensor
        e1.record()
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        t = torch.tensor([e2e_ms], device=dev)
        e2e_rank_ms = [e2e_ms]
        if world > 1:
            allms = [torch.zeros(1, device=dev) for _ in range(world)]
            dist.all_gather(allms, t)
            e2e_rank_ms = [float(x.item()) for x in allms]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_value = B_PER_GPU * world * args.e2e_steps / (float(t.item()) * 1e-3)
        h2d_gbs_per_rank = [round(h2d * args.e2e_steps / (m * 1e-3) / 1e9, 2) for m in e2e_rank_ms]
        del host
        torch.set_num_threads(host_threads)

    secondary = {"ctdet_decode_from_logits": {"value": logit_value, "unit": UNIT,
                                              "note": "same workload, input = pre-sigmoid logits, sigmoid fused "
                                                      "into the selection kernel (one launch, no heat map written)"}}
    if world > 1 and not args.no_secondary:       # collective: every rank takes part (E2, training-side exchange)
        try:
            import bench_secondary
            secondary.update(bench_secondary.run_allreduce(dev, world, rank))
        except Exception as e:
            secondary["grad_allreduce_dla34"] = {"failed": str(e)[:200]}
    if rank == 0 and world == 1 and not args.no_secondary:
        try:
            import bench_secondary
            secondary.update(bench_secondary.run(dev, batches, K=K, steps=min(max(args.steps, 5), 20)))
        except Exception as e:
            secondary["failed"] = str(e)[:200]
    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        # the decode call is ONE kernel launch in this geometry (k_select_hot: NMS + top-K + gathers +
        # box assembly, finalize fused); per-launch time = CUDA-event time of the timed region / steps
        per_launch_s = ms_max * 1e-3 / args.steps
        achieved = ALG_BYTES_PER_IMAGE * B_PER_GPU / per_launch_s / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "per_rank_ms_per_step": [round(m / args.steps, 5) for m in per_rank_ms],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": NCU_TRAFFIC_BYTES, "peak_source": peak_src,
                         "traffic_source": "profiles/r2_select_hot_summary.csv (ncu --set full: "
                                           "dram__bytes_read.sum + dram__bytes_write.sum, one launch)",
                         "kernel": "k_select_hot (the whole decode call is this one launch)",
                         "alg_bytes_per_launch": ALG_BYTES_PER_IMAGE * B_PER_GPU},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps,
                    "h2d_gbs_per_rank": h2d_gbs_per_rank if args.e2e_steps > 0 else None,
                    "h2d_probe_gbs": round(h2d_probe, 2) if args.e2e_steps > 0 else None, "host_binding": numa,
                    "bound_by": "PCIe Gen5 x16 host->device copy of the fp32 heat/wh/reg batch (352 MB per step, "
                                "pinned, chunked and overlapped with the decode); the decode itself is ~1% of it"},
            "gpu_launches": int(launches),
            "secondary": secondary,
            "clocks": sampler.summary(),
            "lib_version": centernet_b200.version(),
        }
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            threads, _ = _calibrate_cpu(cores)
            rate, ts = cpu_port_rate(16, 5, threads)
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                   "sample": "16 images of the same synthetic distribution, median of 5 runs, "
                                             "torch CPU op port of the reference path (oracle/torch_port.py); "
                                             "%d host cores present" % cores}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
