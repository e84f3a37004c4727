#!/usr/bin/env python
"""bench.py -- CCA hot-path benchmark (BASELINE.json metric).

metric  : CCA fwd+bwd pixels/s @ B x 512 x 97 x 97, R=2  (pixels counted once per step; SURVEY.md 8d)
step    : one pass of the hot path over one synthetic batch = the criss-cross attention operator
          (q,k,v -> out forward, dout -> dq,dk,dv backward; cc_attention/functions.py:30-47 and its autograd)
          applied R=2 times in sequence (networks/ccnet.py:118-119), fp32, B=8 images per GPU.  Weak scaling:
          images are sharded across ranks; the op needs no collective.
value   : that op sequence with q,k,v,dout resident in HBM (the boundary SURVEY.md 8(d) defines the
          algorithmic bytes on, so ``roofline`` describes exactly the timed kernels).
e2e     : the same R=2 fwd+bwd through the user-facing drop-in ``cc_attention.CrissCrossAttention`` nn.Module
          (stock-torch 1x1 Q/K/V convs + our op + residual; DDP grad all-reduce when N>1), x from pinned host
          memory every step, y and dx copied back to pinned host memory.  ``module`` = same, x resident.
roofline: all kernels of one op forward / backward (our .so), algorithmic bytes of SURVEY.md 8(d) over the
          CUDA-event time of those launches (L2 flushed between iterations).
--impl reference : the reference module's CPU path (oracle module port; the Python reference cannot
          travel to the GPU box) on the host cores, bounded sample of the same workload.
--dump-outputs DIR : after the timed op steps, rank 0 writes what the last step's last recurrence returned (out, lse, dq,
          dk, dv) as DIR/<name>.npy in float32, for comparing two builds on the same seeded inputs (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(B=8, C=512, H=97, W=97, R=2)
METRIC = "cca_fwd_bwd_pixels_per_s"
UNIT = "pixels/s"


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def shard_images(global_batch: int, rank: int, world: int):
    """Image indices of ``rank`` when ``global_batch`` images are dealt to ``world`` ranks (engine.py:86-88)."""
    per = global_batch // world
    return list(range(rank * per, (rank + 1) * per))


def alg_bytes(B, C, H, W, esize, fwd=True, bwd=True):
    """SURVEY.md 8(d): fwd = s*N*(2Cq+2C), bwd = s*N*(4Cq+4C) per recurrence step."""
    N, Cq = B * H * W, C // 8
    return esize * N * ((2 * Cq + 2 * C) * (1 if fwd else 0) + (4 * Cq + 4 * C) * (1 if bwd else 0))


def bind_to_gpu_numa_node(local_rank: int):
    """Pin this rank's CPU affinity (and with it the first-touch placement of the pinned host buffers it allocates next) to
    the NUMA node its GPU hangs off.  8 ranks x 462 MB/step of pinned copies through one socket's memory controllers is what
    capped the end-to-end curve at 8 GPUs in round 1 (GPUs 4-7 sit on NUMA node 1)."""
    info = {"numa_node": None, "cpus": None}
    try:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = vis.split(",")[local_rank].strip() if vis else str(local_rank)      # nvidia-smi indexes physical devices
        bdf = subprocess.run(["nvidia-smi", "-i", phys, "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:                    # nvidia-smi prints an 8-digit domain, sysfs a 4-digit one
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return info
        cpulist = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        pass
    return info


def ncu_traffic(dtype_name: str):
    """DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) of one op forward / backward, parsed from the committed
    ncu summary of tools/run_op.py (BASELINE config 2, fp32 or bf16).  Returns None when no capture matches."""
    fname = "r02_tc_ncu_summary.txt" if dtype_name == "f32" else "r02_tc_ncu_summary_bf16.txt"
    path = os.path.join(ROOT, "profiles", fname)
    if not os.path.exists(path):
        return None
    units = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}
    tot = {"fwd": 0.0, "bwd": 0.0}
    cur = None
    for line in open(path):
        if line.startswith("Kernel Name"):
            name = line.split(None, 2)[2]
            cur = "fwd" if ("stats_kernel" in name or "fwd_kernel" in name) else ("bwd" if "bwd" in name else None)
        elif cur and (line.startswith("dram__bytes_read.sum") or line.startswith("dram__bytes_write.sum")):
            f = line.split()
            tot[cur] += float(f[1].replace(",", "")) * units.get(f[2].lower(), 1.0)
    if tot["fwd"] == 0.0 or tot["bwd"] == 0.0:
        return None
    return {"fwd": tot["fwd"], "bwd": tot["bwd"], "source": "profiles/" + fname}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_reference_run(steps: int, warmup: int, sample_b: int = 8):
    """The reference module's CPU path (oracle module port, torch CPU ops, all host threads)."""
    from oracle.cca_oracle import CrissCrossAttentionOracle, rcca_forward
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    torch.manual_seed(0)
    C, H, W, R = CFG["C"], CFG["H"], CFG["W"], CFG["R"]
    m = CrissCrossAttentionOracle(C)
    with torch.no_grad():
        m.gamma.fill_(1.0)
    # torch's CPU bmm/conv can get slower with very many threads; give the reference its best thread count
    best = (float("inf"), avail)
    xs = torch.randn(1, C, H, W, requires_grad=True)
    for nt in sorted({n for n in (avail, 64, 32, 16, 8) if n <= avail}, reverse=True):
        torch.set_num_threads(nt)
        for rep in range(2):
            t0 = time.perf_counter()
            rcca_forward(m, xs, R).sum().backward()
            dt = time.perf_counter() - t0
        xs.grad = None
        m.zero_grad(set_to_none=True)
        if dt < best[0]:
            best = (dt, nt)
    cores = best[1]
    torch.set_num_threads(cores)
    x = torch.randn(sample_b, C, H, W, requires_grad=True)
    g = torch.randn(sample_b, C, H, W)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        y = rcca_forward(m, x, R)
        (y * g).sum().backward()
        dt = time.perf_counter() - t0
        x.grad = None
        m.zero_grad(set_to_none=True)
        if it >= warmup:
            times.append(dt)
    total = sum(times)
    return {"value": sample_b * H * W * len(times) / total, "ms_per_step": 1e3 * total / len(times), "cores": cores,
            "host_logical_cpus": avail,
            "sample": f"best of thread counts tried up to {avail} = {cores} threads; B={sample_b} of the B=8 workload ({sample_b}x{C}x{H}x{W}, R={R}, fwd+bwd, fp32), "
                      f"{len(times)} timed steps after {warmup} warm-up"}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    r = cpu_reference_run(max(1, min(args.steps, 5)), max(1, min(args.warmup, 1)))
    line = {"metric": METRIC, "value": r["value"], "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(), "note": "reference module CPU path (oracle port), bounded sample"},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "host_logical_cpus": r["host_logical_cpus"],
                             "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_name():
    return (f"criss-cross attention op x R={CFG['R']} fwd+bwd, B={CFG['B']}/GPU C={CFG['C']} Cq={CFG['C'] // 8} "
            f"{CFG['H']}x{CFG['W']} fp32 (BASELINE configs[1]); e2e/reference arm: the CrissCrossAttention nn.Module "
            f"(1x1 convs + op + residual) on the same shape")


DUMP_MAX_ELEMS = 1 << 21        # per array (8 MB as float32): the five op outputs stay under 64 MB in all


def dump_outputs(path, tensors):
    """Write each tensor as ``path/<name>.npy`` in float32.  A tensor of at most DUMP_MAX_ELEMS elements is written whole in
    its logical (NCHW) shape; a larger one as the 1-D sample ``t.contiguous().view(-1)[idx]`` with
    ``idx = sorted(numpy.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))``, so every run of the
    same shape samples the same elements."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in tensors.items():
        t = t.detach().float().contiguous()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.view(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def time_events(fn, steps, warmup, barrier=None, finish=None):
    """finish(): joins side streams into the current stream before the closing event (pipelined e2e)."""
    for _ in range(warmup):
        fn()
    if finish:
        finish()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if finish:
        finish()
    e1.record()
    torch.cuda.synchronize()
    if barrier:
        barrier()
    return e0.elapsed_time(e1) / steps          # ms per step


def run_ours(args):
    import torch.distributed as dist
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (ccnet_b200 has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)      # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from ccnet_b200 import RCCA, capi, cca_backward, cca_forward
    lib = capi.load()
    assert lib.cca_b200_device_ok() == 1, "not an sm_100 device"

    B, C, H, W, R = CFG["B"], CFG["C"], CFG["H"], CFG["W"], CFG["R"]
    Cq = C // 8
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16}[args.dtype]
    esize = 4 if dtype == torch.float32 else 2
    torch.manual_seed(1234 + rank)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    model = RCCA(C, recurrence=R, impl=args.kernels).to(dev)
    with torch.no_grad():
        model.cca.gamma.fill_(1.0)
    if dtype == torch.bfloat16:
        model = model.to(torch.bfloat16)
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local_rank]) if world > 1 else model

    x_host = torch.randn(B, C, H, W, dtype=dtype).pin_memory()
    g = torch.randn(B, C, H, W, device=dev, dtype=dtype)
    x = x_host.to(dev).requires_grad_(True)
    y_host = torch.empty_like(x_host).pin_memory()
    dx_host = torch.empty_like(x_host).pin_memory()

    def step_resident():
        y = net(x)
        (y * g).sum().backward()
        x.grad = None
        net.zero_grad(set_to_none=True)

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True).requires_grad_(True)
        y = net(xd)
        (y * g).sum().backward()
        y_host.copy_(y.detach(), non_blocking=True)
        dx_host.copy_(xd.grad, non_blocking=True)
        net.zero_grad(set_to_none=True)
        torch.cuda.current_stream().synchronize()

    # Pipelined variant of the same step (what a throughput-minded caller does): the H2D copy of the next step's x and
    # the D2H copies of the previous step's y and dx run on their own streams, overlapped with the compute of the
    # current step.  Every step still moves its own x in and its own y, dx out inside the timed region.
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    x_dev = [torch.empty(B, C, H, W, device=dev, dtype=dtype) for _ in range(2)]
    # results are parked in persistent device buffers (one D2D copy each on the compute stream) so that the D2H stream never
    # holds autograd-owned blocks: no record_stream / caching-allocator interplay, the overlap is deterministic
    y_dev = [torch.empty(B, C, H, W, device=dev, dtype=dtype) for _ in range(2)]
    dx_dev = [torch.empty(B, C, H, W, device=dev, dtype=dtype) for _ in range(2)]
    y_hosts = [y_host, torch.empty_like(x_host).pin_memory()]
    dx_hosts = [dx_host, torch.empty_like(x_host).pin_memory()]
    ev_in = [torch.cuda.Event() for _ in range(2)]          # x_dev[slot] filled
    ev_free = [torch.cuda.Event() for _ in range(2)]        # x_dev[slot] consumed by the compute stream
    ev_res = [torch.cuda.Event() for _ in range(2)]         # y_dev / dx_dev[slot] written by the compute stream
    ev_out = [torch.cuda.Event() for _ in range(2)]         # y_dev / dx_dev[slot] copied out
    pipe = {"i": 0, "primed": False}

    def _prefetch(slot):
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[slot])                  # the step that last read x_dev[slot] has finished
            x_dev[slot].copy_(x_host, non_blocking=True)
            ev_in[slot].record(s_in)

    def step_e2e_pipelined():
        cur = torch.cuda.current_stream()
        slot = pipe["i"] & 1
        if not pipe["primed"]:
            for e in ev_free + ev_out:
                e.record(cur)
            _prefetch(slot)
            pipe["primed"] = True
        _prefetch(slot ^ 1)                                 # next step's input, while this step computes
        cur.wait_event(ev_in[slot])
        xd = x_dev[slot].detach().requires_grad_(True)
        y = net(xd)
        (y * g).sum().backward()
        ev_free[slot].record(cur)
        cur.wait_event(ev_out[slot])                        # the D2H of two steps ago has drained these buffers
        y_dev[slot].copy_(y.detach())
        dx_dev[slot].copy_(xd.grad)
        ev_res[slot].record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_res[slot])
            y_hosts[slot].copy_(y_dev[slot], non_blocking=True)
            dx_hosts[slot].copy_(dx_dev[slot], non_blocking=True)
            ev_out[slot].record(s_out)
        net.zero_grad(set_to_none=True)
        pipe["i"] += 1

    def join_streams():
        cur = torch.cuda.current_stream()
        cur.wait_stream(s_out)
        cur.wait_stream(s_in)

    barrier = (lambda: dist.barrier()) if world > 1 else None

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- operator tensors (resident), in the layout the selected kernels work on ---------------------
    q = torch.randn(B, Cq, H, W, device=dev, dtype=dtype) * 0.58
    k = torch.randn(B, Cq, H, W, device=dev, dtype=dtype) * 0.58
    v = torch.randn(B, C, H, W, device=dev, dtype=dtype) * 0.58
    do = torch.randn(B, C, H, W, device=dev, dtype=dtype)
    from ccnet_b200.functional import tc_eligible
    if args.kernels != "simt" and tc_eligible(B, Cq, C, H, W, dtype):
        # the tensor-core kernels are channels-last; hand them resident tensors in their own layout
        q, k, v, do = (t.contiguous(memory_format=torch.channels_last) for t in (q, k, v, do))
    op_layout = "channels_last" if not q.is_contiguous() else "nchw"

    last = {}                                       # what the latest step returned (for --dump-outputs)

    def step_op():                                  # R sequential op applications, forward + backward
        for _ in range(R):
            out, lse = cca_forward(q, k, v, impl=args.kernels)
            dq, dk, dv = cca_backward(do, q, k, v, out, lse, impl=args.kernels)
        last.update(out=out, lse=lse, dq=dq, dk=dk, dv=dv)

    # ---- main timed region: op level, resident ------------------------------------------------------
    n0 = capi.launch_count()
    with ClockSampler(local_rank) as clk:
        ms = time_events(step_op, args.steps, args.warmup, barrier)
    launches = (capi.launch_count() - n0) * args.steps // (args.steps + args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    ms = max_over_ranks(ms)
    px = B * H * W * world
    value = px / (ms * 1e-3)

    # ---- module level: resident and e2e (host buffers) -----------------------------------------------
    ms_mod = max_over_ranks(time_events(step_resident, max(3, args.steps // 2), 3, barrier))
    module = {"value": px / (ms_mod * 1e-3), "unit": UNIT, "ms_per_step": ms_mod,
              "note": "CrissCrossAttention nn.Module x R fwd+bwd, x resident (NCHW in, converted once per call); projections, "
                      "attention and their backward all on this repository's tcgen05 kernels (one autograd node per step)"}
    ms_e2e_serial = max_over_ranks(time_events(step_e2e, max(3, args.steps // 2), 3, barrier))
    ms_e2e = max_over_ranks(time_events(step_e2e_pipelined, max(6, args.steps // 2), 4, barrier, finish=join_streams))
    e2e = {"value": px / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": x_host.numel() * esize, "d2h_bytes_per_step": 2 * x_host.numel() * esize,
           "serial_ms_per_step": ms_e2e_serial, "serial_value": px / (ms_e2e_serial * 1e-3),
           "note": "nn.Module x R fwd+bwd; every step copies its x from pinned host memory and its y and dx back to pinned "
                   "host memory inside the timed region; value: copies on side streams overlapped with the neighbouring "
                   "steps' compute (double-buffered); serial_*: the same step with copy -> compute -> copy -> sync in sequence",
           "bound": "host link: %.0f MB out + %.0f MB in per step per GPU; at N GPUs the ranks share the host's memory / PCIe "
                    "bandwidth (each rank is bound to its GPU's NUMA node)" % (2 * x_host.numel() * esize / 1e6, x_host.numel() * esize / 1e6),
           "d2h_gbs": 2 * x_host.numel() * esize / (ms_e2e * 1e-3) / 1e9}

    # ---- per-op timings of the kernels of this repo -> roofline ----------------------------------------
    out, lse = cca_forward(q, k, v, impl=args.kernels)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > L2 (126 MB)

    def op_time(fn, iters=10):
        ts = []
        for _ in range(3):
            fn()
        for _ in range(iters):
            flush.zero_()
            torch.cuda._sleep(300000)          # ~0.15 ms of GPU spin: the host enqueues the op's launches meanwhile, so the
                                               # events bracket back-to-back kernels, not host launch latency
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return sum(ts) / len(ts), ts[0]

    n1 = capi.launch_count()
    f_avg, f_min = op_time(lambda: cca_forward(q, k, v, impl=args.kernels))
    nf = (capi.launch_count() - n1) // 13
    n1 = capi.launch_count()
    b_avg, b_min = op_time(lambda: cca_backward(do, q, k, v, out, lse, impl=args.kernels))
    nb = (capi.launch_count() - n1) // 13
    peak, peak_src = measured_peaks()
    bytes_f, bytes_b = alg_bytes(B, C, H, W, esize, True, False), alg_bytes(B, C, H, W, esize, False, True)
    dom_is_bwd = b_avg >= f_avg
    dom_bytes, dom_ms = (bytes_b, b_avg) if dom_is_bwd else (bytes_f, f_avg)
    ach = dom_bytes / (dom_ms * 1e-3) / 1e9
    # DRAM traffic of one op call: parsed from the committed ncu --set full summary of tools/run_op.py (same shape / dtype)
    traffic = None
    if (B, C, H, W) == (8, 512, 97, 97) and op_layout == "channels_last":
        traffic = ncu_traffic("f32" if dtype == torch.float32 else "bf16")
    roofline = {"bound": "hbm", "kernel": "cca backward op (prep + one persistent item kernel)" if dom_is_bwd
                else "cca forward op (statistics pre-pass + values kernel)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": (traffic["bwd" if dom_is_bwd else "fwd"] if traffic else None),
                "traffic_fwd": traffic["fwd"] if traffic else None, "traffic_bwd": traffic["bwd"] if traffic else None,
                "traffic_source": (traffic["source"] + " (ncu --set full; sum over the launches of one op call)") if traffic else None,
                "peak_source": peak_src, "launches_per_op": nb if dom_is_bwd else nf,
                "op_fwd": {"ms": f_avg, "ms_min": f_min, "alg_bytes": bytes_f, "gbs": bytes_f / f_avg / 1e6,
                           "frac": bytes_f / f_avg / 1e6 / peak, "launches": nf},
                "op_bwd": {"ms": b_avg, "ms_min": b_min, "alg_bytes": bytes_b, "gbs": bytes_b / b_avg / 1e6,
                           "frac": bytes_b / b_avg / 1e6 / peak, "launches": nb},
                "op_layout": op_layout,
                "timing": "CUDA events on torch's current stream (the launching stream), L2 flushed between iterations"}

    # ---- the same op in the other I/O dtype (BASELINE config 2: "fp32 vs bf16"), operator-only ---------------------------
    other = None
    if rank == 0:
        odt = torch.bfloat16 if dtype == torch.float32 else torch.float32
        oes = 2 if odt == torch.bfloat16 else 4
        fmt = torch.channels_last if tc_eligible(B, Cq, C, H, W, odt) and args.kernels != "simt" else torch.contiguous_format
        q2, k2, v2, do2 = (t.to(odt).contiguous(memory_format=fmt) for t in (q, k, v, do))
        out2, lse2 = cca_forward(q2, k2, v2, impl=args.kernels)
        f2, _ = op_time(lambda: cca_forward(q2, k2, v2, impl=args.kernels), iters=6)
        b2, _ = op_time(lambda: cca_backward(do2, q2, k2, v2, out2, lse2, impl=args.kernels), iters=6)
        bf2, bb2 = alg_bytes(B, C, H, W, oes, True, False), alg_bytes(B, C, H, W, oes, False, True)
        other = {"dtype": "bf16" if odt == torch.bfloat16 else "f32",
                 "op_fwd": {"ms": f2, "alg_bytes": bf2, "gbs": bf2 / f2 / 1e6, "frac": bf2 / f2 / 1e6 / peak},
                 "op_bwd": {"ms": b2, "alg_bytes": bb2, "gbs": bb2 / b2 / 1e6, "frac": bb2 / b2 / 1e6 / peak},
                 "op_fwd_bwd_pixels_per_s_R2": B * H * W / (R * (f2 + b2) * 1e-3),
                 "layout": "channels_last" if fmt == torch.channels_last else "nchw"}
        del q2, k2, v2, do2, out2, lse2
    roofline["other_dtype"] = other

    # ---- the network around the operator (BASELINE configs[2], [3]): ResNet101+RCCA, synthetic 769x769, global batch 8 ----
    ccnet = None
    if not args.no_train:
        del x, g, x_dev, y_dev, dx_dev, q, k, v, do, out, lse, flush
        torch.cuda.empty_cache()
        from harness.train_synth import run as train_run
        try:
            ccnet = train_run(local_rank, world, steps=max(2, min(args.steps, 4)), warmup=2, allow_tf32=True)
            ccnet["note"] = ("train step = the reference's loop (train.py:199-239) on synthetic data, stock torch backbone (cudnn, TF32 "
                             "convolutions = torch default), DDP + SyncBatchNorm when N > 1, per-GPU batch = 8 / N (engine.py:88); "
                             "cca_modules_ms = the R criss-cross modules alone (projection GEMMs + operator + residual, fwd+bwd) "
                             "at the head's feature-map size")
            if world == 1:                            # evaluate.py's loop on one synthetic Cityscapes-sized image (8 windows of 769^2)
                torch.cuda.empty_cache()
                from harness.eval_synth import run as eval_run
                ccnet["eval"] = eval_run(local_rank, steps=1, warmup=1)
        except Exception as exc:                      # never lose the main line to the extra leg
            ccnet = (ccnet or {}) | {"error": repr(exc)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_reference_run(3, 1)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "host_logical_cpus": r["host_logical_cpus"],
               "kind": "port", "sample": r["sample"]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32" if dtype == torch.float32 else "bf16", "data": "synthetic",
                "config": {"workload": workload_name(), "global_batch": B * world, "kernels": args.kernels,
                           "op_layout": op_layout,
                           "l2": "inputs larger than L2: one op fwd+bwd touches q,k,v,dout,out,dq,dk,dv = 1.04 GB vs 126 MB "
                                 "L2 (no explicit flush in the timed loop); the per-op roofline timings flush 256 MB explicitly",
                           "parallelism": f"dp{world} (image-sharded, DDP grad all-reduce only)",
                           "host_binding": numa},
                "clocks": clk.summary(), "e2e": e2e, "module": module, "gpu_launches": int(launches),
                "roofline": roofline, "ccnet": ccnet, "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--kernels", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-train", action="store_true", help="skip the ResNet101+RCCA train-step leg (BASELINE configs[2], [3])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed op step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
