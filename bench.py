#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Enoki backend.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (N=1 and every rank of N>1, weak scaling): BASELINE.json configs[1] =
"CUDAArray<float> 64M-elem fused arith+exp/sin chain, cuda_eval()":
    t = fmadd(x0,x1,x2); u = exp(-(t*t)); v = sin(fmadd(x3,u,x0)); out = fmadd(v,x1,sqrt(abs(t)))
on N = 2^26 fp32 elements per GPU (SURVEY.md 8d, C2).  One step = record the expression through
the C ABI, cuda_eval() it (one fused sweep kernel: 4 input streams + 1 output stream = 20 B/elem),
plus a fused hsum of the output whose scalar is all-reduced over NCCL when N>1 (the only
cross-GPU value, SURVEY 8e).  Metric: M array-ops/s (DAG nodes x elements / s, jit.cu:1219-1222).

The JSON line also carries
  roofline      -- the sweep kernel's algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json; names the kernel
                   that ran (fast or general: ek_init()'s kernel qualification decides) and what the qualification timed
  backward      -- the C4 tape (10 240 nodes / 20 224 edges, node width 131 072): M edge-adjoints/s
  e2e           -- same metric through the C ABI with pinned HOST buffers (H2D + D2H inside the timing), with the PCIe
                   ceiling of the same copies beside it
  cpu_baseline  -- the reference's own CPU path (oracle/_ref) timed on this box's host cores
  histogram     -- C3 (configs[2]): 2^26-sample gather + scatter_add histogram, kernel time
  c5            -- configs[4]: 4096^2 differentiable ray-sphere render, forward + backward (tools/c5_bench, C++ header API)
  c1_cpu        -- configs[0]: the reference's CPU path alone, a*b+sin(c) at 2^20, operator form and vectorize() form
  backward_width_16384 -- the C4 tape at node width 16 384 (host-limited regime)
  small         -- the C2 expression on 2^20 elements (launch-latency regime)
  clocks        -- nvidia-smi SM clock / throttle reasons sampled inside the timed window
`--impl reference` times the reference CPU path alone (rank 0 only).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ELEMS = 1 << 26
C2_NODES = 9            # fma, mul, neg, exp, fma, sin, abs, sqrt, fma (what the runtime counts as ops=)
C2_BYTES_PER_ELEM = 20  # 4 input streams + 1 output stream, fp32 (SURVEY 8d)
C4 = dict(levels=80, per_level=128, width=131072)
DUMP_ELEMS = 1 << 22    # --dump-outputs: at most 16 MiB of float32 output


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Sample nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.proc = None
        self.device = device
        self.lines = []
        self.t_lines = []
        self.window = [None, None]

    def start(self):
        """Starts `nvidia-smi -lms 100` and waits (<= 5 s) for its first line, so that samples exist during the
        timed region and not only after it."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.device)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        first = threading.Event()

        def reader():
            for line in self.proc.stdout:
                self.lines.append(line); self.t_lines.append(time.time())
                first.set()
        self.thread = threading.Thread(target=reader, daemon=True)
        self.thread.start()
        first.wait(5.0)

    def mark_begin(self): self.window[0] = time.time()
    def mark_end(self): self.window[1] = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.thread.join(timeout=2)
        lines = list(self.lines)
        n_all = len(lines)
        window_note = "timed region"
        if self.window[0] is not None and self.window[1] is not None:
            inside = [l for l, t in zip(lines, self.t_lines) if self.window[0] <= t <= self.window[1] + 0.1]
            if len(inside) < 3:
                # a short timed region (a few ms at --steps 20) holds less than three 25 ms samples: widen by half a second on
                # both sides -- the warm-up steps before and the kernel-timing pass after it keep the GPU under the same load
                inside = [l for l, t in zip(lines, self.t_lines) if self.window[0] - 0.5 <= t <= self.window[1] + 0.5]
                window_note = "timed region +- 0.5 s (warm-up / kernel-timing pass, same load)"
            if inside:
                lines = inside
        out = "".join(lines)
        sm, smax, reasons = [], None, set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            # the timed region was shorter than one sampling period: take one sample now (still warm)
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.device)],
                                     capture_output=True, text=True, timeout=10).stdout
                f = [x.strip() for x in out.strip().split(",")]
                sm.append(float(f[1])); smax = float(f[2])
            except Exception:
                pass
        busy = [v for v in sm if smax and v >= 0.5 * smax] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "samples_whole_run": n_all, "window": window_note}


# --------------------------------------------------------------------------- reference CPU arm
def load_ref(fast=True):
    name = "libenoki_ref_fast.so" if fast else "libenoki_ref.so"
    path = os.path.join(ROOT, "oracle", "_ref", name)
    if os.path.exists(path):
        lib = ctypes.CDLL(path)
        lib.ref_c2_time.restype = ctypes.c_double
        lib.ref_c2_time_vectorized.restype = ctypes.c_double
        lib.ref_info.restype = ctypes.c_char_p
        return lib, "reference"
    path = os.path.join(ROOT, "oracle", "liboracle.so")
    lib = ctypes.CDLL(path)
    lib.or_c2_time.restype = ctypes.c_double
    return lib, "port"


def aligned_f32(n, align=64):
    """float32 buffer whose address is `align`-byte aligned (DynamicArray::map needs packet alignment)."""
    raw = np.zeros(n * 4 + align, np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + n * 4].view(np.float32)


class CpuC2:
    """The reference's CPU implementation of C2 on `threads` host threads, each on its own slice of
    `sample_elems` elements (Enoki is single-threaded by construction; the split is the embarrassingly
    parallel one of BASELINE.md section 3).  Buffers are allocated once; run() returns elements/s."""

    def __init__(self, sample_elems, threads):
        self.lib, self.kind = load_ref(True)
        self.threads = threads
        self.per = (sample_elems // threads) // 16 * 16
        rng = np.random.default_rng(0)
        block = rng.uniform(-4, 4, min(self.per, 1 << 20)).astype(np.float32)
        self.bufs = []
        for _ in range(threads):
            xs = []
            for k in range(4):
                a = aligned_f32(self.per)
                for o in range(0, self.per, len(block)):
                    m = min(len(block), self.per - o)
                    a[o:o + m] = np.roll(block, 17 * k + 1)[:m]
                xs.append(a)
            self.bufs.append((xs, aligned_f32(self.per)))

    def run(self, reps):
        best = [0.0] * self.threads
        per = self.per

        def work(t):
            xs, out = self.bufs[t]
            if self.kind == "reference":
                # the reference's own fastest CPU form: the fused vectorize() loop (dynamic.h:1025-1074)
                best[t] = self.lib.ref_c2_time_vectorized(P(xs[0]), P(xs[1]), P(xs[2]), P(xs[3]), P(out), ctypes.c_size_t(per), reps)
            else:
                best[t] = self.lib.or_c2_time(P(xs[0]), P(xs[1]), P(xs[2]), P(xs[3]), P(out), ctypes.c_size_t(per), reps)

        ths = [threading.Thread(target=work, args=(t,)) for t in range(self.threads)]
        for th in ths: th.start()
        for th in ths: th.join()
        return per * self.threads / max(best)


def host_cores():
    """Cores this process may really use: min(affinity mask, cgroup CPU quota).  The GPU boxes expose 128 logical CPUs
    but the container is capped (cpu.max = 16 CPUs); threads beyond the quota only get throttled."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return n


def cpu_wall_rate(c, passes):
    """elements/s of CpuC2 `c` by the wall clock around thread start and join (not the per-thread best pass, which is
    blind to CPU-quota throttling)."""
    t0 = time.time()
    c.run(passes)
    return passes * c.per * c.threads / (time.time() - t0)


def best_cpu_config(sample_elems):
    """The reference CPU path on the thread count that is fastest by the wall clock (quota cores, or twice that)."""
    cores = host_cores()
    best = None
    for th in sorted({cores, min(2 * cores, os.cpu_count() or cores)}):
        c = CpuC2(sample_elems, th)
        c.run(1)
        r = cpu_wall_rate(c, 4)
        if best is None or r > best[1]:
            best = (c, r)
    return best[0], cores


def cpu_c2(sample_elems, reps, threads):
    c = CpuC2(sample_elems, threads)
    t0 = time.time()
    r = c.run(reps)
    return r, c.kind, time.time() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = N_ELEMS              # the whole 2^26-element workload, split over the host threads (DRAM resident)
    c, quota = best_cpu_config(sample)
    cores = c.threads
    for _ in range(max(args.warmup, 1)):
        c.run(1)
    # K timed "steps": each step = PASSES passes of the whole 2^26-element workload on all host threads, timed by the
    # wall clock around thread start and join (what a caller of the reference would see; the passes amortise the
    # thread start-up).  value and ms_per_step come from the same clock.
    t_pass = (c.per * c.threads) / cpu_wall_rate(c, 2)           # seconds per pass, measured (incl. thread start / 2)
    PASSES = int(max(1, min(32, round(60.0 / (max(args.steps, 1) * t_pass)))))   # whole timed run <= ~1 minute
    t0 = time.time()
    for _ in range(args.steps):
        c.run(PASSES)
    wall = time.time() - t0
    elems_per_s = args.steps * PASSES * (c.per * c.threads) / wall
    value = elems_per_s * C2_NODES / 1e6
    line = {
        "impl": "reference", "metric": "M array-ops/s (eval)", "value": value, "unit": "M array-ops/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: CUDAArray<float> 64M-elem fused arith+exp/sin chain (CPU: DynamicArray<Packet<float,8>> vectorize() form)",
                   "elems": N_ELEMS, "nodes": C2_NODES},
        "cpu_baseline": {"value": value, "unit": "M array-ops/s", "cores": cores, "kind": c.kind,
                         "sample": f"{PASSES} passes over all {sample} elements per step, split over {cores} threads (host exposes {os.cpu_count()} CPUs, CPU quota {quota}; DRAM resident), vectorize() form, AVX2+FMA -ffp-contract=fast, wall clock incl. thread start"},
        "e2e": {"value": value, "unit": "M array-ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--elems", type=int, default=N_ELEMS, help="elements per GPU (default: the BASELINE config, 2^26)")
    ap.add_argument("--skip-backward", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling aid: leave out the host-buffer leg")
    ap.add_argument("--skip-extras", action="store_true", help="profiling aid: leave out C3 / small / C5 / C1 objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy: out.npy (float32; the "
                         f"whole output up to {DUMP_ELEMS} elements, beyond that the elements at a fixed seeded sample of "
                         "indices) and hsum.npy (the loss scalar, all-reduced when N>1); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    os.environ.setdefault("NCCL_DEBUG", "WARN")   # never override the caller's setting (NCCL logs go to stderr anyway)
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import enoki_b200 as ek
    from enoki_b200 import Float32, fmadd, exp, sin, sqrt, hsum
    L = ek.lib()
    if L.ek_device_count() == 0:
        raise SystemExit("bench.py: no CUDA device visible -- enoki_b200 has no CPU fallback")
    L.ek_set_device(local_rank)
    assert L.ek_init() == 0, L.ek_last_error()
    torch.cuda.set_device(local_rank)
    ext_stream = torch.cuda.ExternalStream(L.ek_stream(), device=torch.device("cuda", local_rank))

    n = args.elems
    # ---- synthetic inputs, generated on the device by the backend itself (resident in HBM)
    idx = ek.UInt32.arange(n)

    def mk(k):
        h = idx * np.uint32(2654435761 + 2 * k) + np.uint32(12345 * (k + 1) + rank)
        return fmadd(Float32(h >> 8), Float32(8.0 / (1 << 24)), Float32(-4.0))
    x = [mk(k) for k in range(4)]
    ek.cuda_eval(); ek.cuda_sync()
    del idx

    native_nccl = False
    # EK_BENCH_NATIVE_NCCL=1: the per-step all-reduce through the library's own communicator (C ABI, csrc/ek_dist.cpp).
    # Off by default in round 2: that path has not run on hardware yet, the torch.distributed one has (round 1, N=2).
    if world > 1 and os.environ.get("EK_BENCH_NATIVE_NCCL") == "1":
        try:
            from enoki_b200.dist import init_native
            native_nccl = init_native(rank, world, torch.device("cuda", local_rank))
        except Exception as e:
            print(f"bench.py: native NCCL path unavailable: {e!r}", file=sys.stderr)

    class DevScalar:
        """expose a 4-byte device buffer to torch (NCCL all-reduce of the loss scalar)"""
        def __init__(self, ptr):
            self.__cuda_array_interface__ = {"shape": (1,), "typestr": "<f4", "data": (ptr, False), "version": 3}

    def step(reduce_scalar=True):
        t = fmadd(x[0], x[1], x[2])
        u = exp(-(t * t))
        v = sin(fmadd(x[3], u, x[0]))
        out = fmadd(v, x[1], sqrt(abs(t)))
        del t, u, v
        s = hsum(out) if reduce_scalar else None
        ek.cuda_eval()
        if world > 1 and s is not None:
            if native_nccl:         # one ncclAllReduce enqueued by the library on its own stream (csrc/ek_dist.cpp)
                from enoki_b200.dist import allreduce_handles
                allreduce_handles([s])
            else:                   # round-1 path: torch.distributed on the backend's stream
                from enoki_b200.dist import allreduce_device_scalar
                allreduce_device_scalar(L.ek_var_ptr(s.index), "f32", L.ek_stream(), torch.device("cuda", local_rank))
        return out, s

    def barrier():
        ek.cuda_sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # runs through warm-up, the timed region and the kernel-timing pass
    for _ in range(args.warmup):
        step()
    barrier()
    L.ek_stats_reset()
    barrier()
    sampler.mark_begin()
    L.ek_timer_start()
    t0 = time.time()
    keep = None
    for _ in range(args.steps):
        keep = step()
    ms = L.ek_timer_stop()
    barrier()
    sampler.mark_end()
    wall_ms = 1e3 * (time.time() - t0)
    st = ek.stats()
    launches = int(st.launches)
    if dist is not None:
        tt = torch.tensor([ms], device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    ms_per_step = ms / args.steps
    value = world * n * C2_NODES / (ms_per_step * 1e-3) / 1e6
    loss_val = float(keep[1].numpy()[0])
    dump = None
    if args.dump_outputs and rank == 0:
        dump = {"out": sample_output(keep[0].numpy()), "hsum": keep[1].numpy().astype(np.float32)}
    del keep

    # ---- roofline of the dominant kernel: per-launch CUDA events on the launch stream
    L.ek_set_timing(1)
    L.ek_stats_reset()
    for _ in range(5):
        o, s = step(reduce_scalar=False)
        del o, s
    stt = ek.stats()
    L.ek_set_timing(0)
    clocks = sampler.stop() if rank == 0 else None
    kern_ms = stt.total_kernel_ms / max(int(stt.sweep_launches), 1)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    achieved = C2_BYTES_PER_ELEM * n / (kern_ms * 1e-3) / 1e9
    on_fast = int(stt.fast_launches) > 0         # which sweep kernel really ran (ek_init's kernel qualification decides)
    traffic, traffic_src = None, None
    if not on_fast and n == (1 << 26):
        # DRAM bytes of one launch of the general kernel from the committed `ncu --set full` capture of this workload
        try:
            traffic_src = "profiles/r1_final_sweep_ncu_summary.txt"
            txt = open(os.path.join(ROOT, traffic_src)).read()
            import re
            rd = re.search(r"dram__bytes_read\.sum \[(\w+)\] = ([0-9.]+)", txt); wr = re.search(r"dram__bytes_write\.sum \[(\w+)\] = ([0-9.]+)", txt)
            unit = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
            traffic = float(rd.group(2)) * unit[rd.group(1)] + float(wr.group(2)) * unit[wr.group(1)]
        except Exception:
            traffic, traffic_src = None, None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                "traffic": traffic, "traffic_unit": "B/launch", "traffic_source": traffic_src if traffic is not None else
                "none: no ncu capture of ek_fast_kernel exists (the repository had no GPU access after the kernel was written)",
                "algorithmic_bytes": C2_BYTES_PER_ELEM * n,
                "kernel": "ek_fast_kernel<256> (ek_sweep_fast.cu)" if on_fast else "ek_sweep_kernel<16,false,true> (ek_sweep.cu)",
                "fast_kernel_qualified": bool(L.ek_fast_mode()), "qualification_timing": _qualification_timing(), "kernel_ms": kern_ms,
                "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "B200_PROFILING.md fallback (of fallback)"}

    # ---- e2e: pinned host buffers, H2D of the 4 inputs + D2H of the result inside the timed region
    e2e = None
    if (rank == 0 or world > 1) and not args.skip_e2e:
        hb = [L.ek_host_malloc(n * 4) for _ in range(5)]
        for k in range(4):
            L.ek_memcpy_from_device(hb[k], L.ek_var_ptr(x[k].index), n * 4)

        E2E_CHUNKS = 8          # the step is pipelined: H2D of chunk c+1 overlaps with the read-back of chunk c

        def e2e_step():
            cn = n // E2E_CHUNKS
            hold = []           # device arrays stay allocated until the read-backs have finished (ek_sync below)
            for c in range(E2E_CHUNKS):
                xs = []
                for k in range(4):
                    d = L.ek_malloc(cn * 4)
                    L.ek_memcpy_to_device_async(d, hb[k] + c * cn * 4, cn * 4)
                    xs.append(Float32.map(d, cn, True))
                t = fmadd(xs[0], xs[1], xs[2])
                out = fmadd(sin(fmadd(xs[3], exp(-(t * t)), xs[0])), xs[1], sqrt(abs(t)))
                del t
                ek.cuda_eval()
                L.ek_memcpy_from_device_overlapped(hb[4] + c * cn * 4, L.ek_var_ptr(out.index), cn * 4)
                hold.append((xs, out))
            ek.cuda_sync()
            del hold

        e2e_steps = max(3, min(args.steps, 5))
        e2e_step()
        barrier()
        te = time.time()
        for _ in range(e2e_steps):
            e2e_step()
        ek.cuda_sync()
        e2e_ms = 1e3 * (time.time() - te) / e2e_steps
        if dist is not None:
            tt = torch.tensor([e2e_ms], device=f"cuda:{local_rank}")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_ms = float(tt.item())
        e2e = {"value": world * n * C2_NODES / (e2e_ms * 1e-3) / 1e6, "unit": "M array-ops/s",
               "h2d_bytes_per_step": 4 * n * 4, "d2h_bytes_per_step": n * 4, "ms_per_step": e2e_ms,
               "pipeline": f"{E2E_CHUNKS} chunks; H2D + kernels on the compute stream, read-back on a second stream",
               "pcie_gbs": (5 * n * 4) / (e2e_ms * 1e-3) / 1e9}
        # PCIe ceiling beside it: the same bytes (4 inputs up, 1 result down) with NO kernels in between -- uploads on the
        # compute stream, the read-back of the previous chunk on the second stream, pinned buffers, same chunking
        try:
            cn = n // E2E_CHUNKS
            dbuf = [L.ek_malloc(cn * 4) for _ in range(5)]

            def copies_only():
                for c in range(E2E_CHUNKS):
                    for k in range(4):
                        L.ek_memcpy_to_device_async(dbuf[k], hb[k] + c * cn * 4, cn * 4)
                    L.ek_memcpy_from_device_overlapped(hb[4] + c * cn * 4, dbuf[4], cn * 4)
                ek.cuda_sync()
            copies_only()
            tc = time.time()
            for _ in range(3):
                copies_only()
            ceil_ms = 1e3 * (time.time() - tc) / 3
            for d in dbuf:
                L.ek_free(d)
            e2e["pcie_ceiling_ms"] = ceil_ms
            e2e["pcie_ceiling_gbs"] = (5 * n * 4) / (ceil_ms * 1e-3) / 1e9
            e2e["frac_of_pcie_ceiling"] = ceil_ms / e2e_ms
        except Exception as e:
            e2e["pcie_ceiling_error"] = repr(e)
        for p in hb:
            L.ek_host_free(p)

    # ---- C3 (configs[2]): 2^26-sample gather + scatter_add histogram, kernel-only time
    hist = None
    if rank == 0 and not args.skip_extras:
        try:
            hist = bench_histogram(ek, L, n, peak_gbs)
        except Exception as e:                      # secondary objects must never cost the headline line
            hist = {"error": repr(e)}

    # ---- launch-latency regime (SURVEY 8d): the same C2 expression on 2^20 elements
    small = None
    if rank == 0 and not args.skip_extras:
      try:
        ns = 1 << 20
        xs_s = [Float32.copy(np.random.default_rng(k).uniform(-4, 4, ns).astype(np.float32)) for k in range(4)]

        def small_step():
            t = fmadd(xs_s[0], xs_s[1], xs_s[2])
            o = fmadd(sin(fmadd(xs_s[3], exp(-(t * t)), xs_s[0])), xs_s[1], sqrt(abs(t)))
            del t
            ek.cuda_eval()
            return o
        for _ in range(5):
            small_step()
        ek.cuda_sync()
        L.ek_timer_start()
        reps_s = 200
        for _ in range(reps_s):
            small_step()
        ms_s = L.ek_timer_stop() / reps_s
        small = {"workload": "C2 on 2^20 elements (launch-latency regime)", "ms_per_step": ms_s,
                 "m_array_ops_per_s": ns * C2_NODES / (ms_s * 1e-3) / 1e6}
        del xs_s
      except Exception as e:
        small = {"error": repr(e)}

    # ---- backward: C4 tape (per rank), K' passes of backward(free_graph=False)
    backward = None
    if not args.skip_backward:
        backward = bench_backward(ek, L, rank, world, dist, torch, local_rank, peak_gbs)

    backward_narrow = None
    if not args.skip_backward and rank == 0 and not args.skip_extras:
        try:        # the same tape at node width 16 384: the regime where the host walk, not HBM, limits backward()
            backward_narrow = bench_backward(ek, L, rank, 1, None, torch, local_rank, peak_gbs, width=16384)
        except Exception as e:
            backward_narrow = {"error": repr(e)}

    # ---- C5 (configs[4]): differentiable ray-sphere render through the C++ header API (tools/c5_bench.cpp)
    c5 = None
    if rank == 0 and not args.skip_extras:
        c5 = bench_c5(peak_gbs, local_rank)

    # ---- C1 (configs[0]): the reference's CPU path alone, operator form and vectorize() form at 2^20
    c1 = None
    if rank == 0 and not args.skip_cpu:
        c1 = bench_c1()

    # ---- CPU baseline beside it (rank 0, bounded sample)
    cpu = None
    if rank == 0 and not args.skip_cpu:
      try:
        c, quota = best_cpu_config(N_ELEMS)
        r = cpu_wall_rate(c, 16)
        single = CpuC2(1 << 24, 1); single.run(1)
        r1 = cpu_wall_rate(single, 2)
        cpu = {"value": r * C2_NODES / 1e6, "unit": "M array-ops/s", "cores": c.threads, "kind": c.kind,
               "sample": f"16 passes over all 2^26 elements split over {c.threads} threads (host exposes {os.cpu_count()} CPUs, CPU quota "
                         f"{quota}; DRAM resident; reference vectorize() form, AVX2+FMA -ffp-contract=fast; wall clock); "
                         f"single thread on 2^24: {r1 * C2_NODES / 1e6:.1f} M array-ops/s"}
      except Exception as e:
        cpu = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": "M array-ops/s (eval)", "value": value, "unit": "M array-ops/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C2: CUDAArray<float> 64M-elem fused arith+exp/sin chain, cuda_eval() (+ fused hsum, NCCL all-reduce of the scalar when N>1)",
                       "elems_per_gpu": n, "nodes": C2_NODES, "bytes_per_elem": C2_BYTES_PER_ELEM,
                       "l2": "inputs 4 x 256 MiB per step exceed the 126 MB L2 (no explicit flush needed)",
                       "parallelism": f"element-range sharding x{world}, one rank per GPU",
                       "collective": ("ncclAllReduce of the loss scalar by the library (C ABI ek_allreduce_scalars)" if native_nccl else
                                      "torch.distributed all_reduce of the loss scalar on the backend's stream") if world > 1 else "none (1 GPU)"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "backward": backward, "backward_width_16384": backward_narrow, "histogram": hist, "c5": c5, "c1_cpu": c1, "small": small, "wall_ms_per_step": wall_ms / args.steps, "loss_checksum": loss_val,
        }
        print(json.dumps(line), flush=True)
    if dump is not None:
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def sample_output(a):
    """`a` itself when it has at most DUMP_ELEMS elements, else its elements at DUMP_ELEMS-or-fewer fixed indices (seeded,
    ascending, depending only on len(a)), so that two builds run with the same arguments dump comparable files."""
    if len(a) <= DUMP_ELEMS:
        return a
    idx = np.unique(np.random.default_rng(0).integers(0, len(a), DUMP_ELEMS))
    return a[idx]


def _qualification_timing():
    """What enoki_b200/ek_qualify measured when ek_init() qualified the fast kernel on this machine (general vs fast kernel,
    C2 and C3 at 2^24 elements, device time of the sweep launch); None when the qualification was skipped or failed earlier."""
    try:     # written by ek_init() (csrc/ek_runtime.cpp) into the temporary directory
        tmp = os.environ.get("TMPDIR") or "/tmp"
        return json.load(open(os.path.join(tmp, f"ek_b200_fast_timing_{os.getuid()}.json")))
    except Exception:
        return None


def bench_c5(peak_gbs, local_rank):
    """BASELINE configs[4] (SURVEY 8d C5): 4096 x 4096 differentiable ray-sphere render, forward + backward, written against
    enoki::DiffArray<enoki::CUDAArray<float>> (tools/c5_bench.cpp, built in the dev container against the reference's API
    headers).  Runs as a child process on the same GPU after this process has finished its own timing; reports ms per
    forward+backward step, the bytes the launched kernels streamed with graph simplification on / off, and those bytes
    against the measured HBM peak.  (Parity of this render against the reference CPU tape: tests/cpp/sphere_check.cpp.)"""
    exe = os.path.join(ROOT, "tools", "c5_bench")
    if not os.path.exists(exe):
        return {"error": "tools/c5_bench is not built (needs the reference headers at build time: __graft_entry__.build())"}
    try:
        env = dict(os.environ, LOCAL_RANK=str(local_rank))
        r = subprocess.run([exe, "4096", "5"], capture_output=True, text=True, timeout=600, env=env)
        if r.returncode != 0:
            return {"error": f"c5_bench rc={r.returncode}: {r.stderr[-400:]}"}
        d = json.loads(r.stdout.strip().splitlines()[-1])
        for key in ("simplify_on", "simplify_off"):
            o = d.get(key)
            if o:
                total = o["sweep_bytes_per_step"] + o["adjoint_bytes_per_step"]
                o["bytes_streamed_per_step"] = total
                o["roofline"] = {"bound": "hbm", "achieved": total / (o["ms_per_step"] * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                                 "frac": total / (o["ms_per_step"] * 1e-3) / 1e9 / peak_gbs,
                                 "note": "bytes the launched kernels streamed (sweep loads + stores, 10 B per edge-adjoint) over the wall "
                                         "time of one traced forward+backward step incl. host tracing; SURVEY 8d nominal: forward 201 MB"}
        d["n_gpus"] = 1
        return d
    except Exception as e:
        return {"error": repr(e)}


def bench_c1():
    """BASELINE configs[0] (SURVEY 8d C1): r = a*b + sin(c) on DynamicArray<Packet<float,8>>, N = 2^20 -- the reference's own
    CPU path (oracle/_ref), operator form and vectorize() form, one thread (Enoki's CPU arrays are single-threaded)."""
    try:
        lib, kind = load_ref(True)
        if kind != "reference":
            return {"error": "oracle/_ref is not built"}
        out = (ctypes.c_float * 1)()
        n = 1 << 20
        res = {"workload": "C1: DynamicArray<Packet<float,8>> 1M-elem a*b+sin(c), AVX2+FMA -ffp-contract=fast, 1 thread, best of 50",
               "elems": n, "nproc": os.cpu_count(), "cpu_quota": host_cores()}
        for name in ("operator", "vectorized"):
            f = getattr(lib, f"ref_c1_time_{name}")
            f.restype = ctypes.c_double
            t = f(ctypes.c_size_t(n), 50, out)
            res[name] = {"ms": t * 1e3, "m_elems_per_s": n / t / 1e6, "m_array_ops_per_s": 3 * n / t / 1e6,
                         "gb_per_s": 16.0 * n / t / 1e9}
        try:
            res["cpu_model"] = next(l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name"))
        except Exception:
            pass
        return res
    except Exception as e:
        return {"error": repr(e)}


def bench_histogram(ek, L, n, peak_gbs):
    """SURVEY 8d C3: samples resident in HBM; idx = UInt32((y+4)*31/8); mask = idx<31; w = gather(table31, idx, mask);
    scatter_add(bins_u32, 1, idx, mask); scatter_add(hist_f32, w, idx, mask).  Algorithmic bytes: 4 B / sample."""
    from enoki_b200 import Float32, UInt32, fmadd, gather, scatter_add
    i = UInt32.arange(n)
    h = i * np.uint32(2654435761) + np.uint32(974711)
    h = (h ^ (h >> 15)) * np.uint32(2246822519)
    y = fmadd(Float32(h >> 8), Float32(8.2 / (1 << 24)), Float32(-4.1))
    ek.cuda_eval(); del i, h
    table = Float32.copy(np.linspace(0.5, 1.5, 31, dtype=np.float32))
    table.eval()

    def one():
        idx = UInt32((y - (-4.0)) * 31.0 / 8.0)
        mask = idx < UInt32(31)
        w = gather(Float32, table, idx, mask)
        bins = UInt32.zero(31); hist = Float32.zero(31)
        scatter_add(bins, UInt32(1), idx, mask)
        scatter_add(hist, w, idx, mask)
        del idx, mask, w
        ek.cuda_eval()
        return bins, hist
    for _ in range(3):
        one()
    L.ek_set_timing(1); L.ek_stats_reset()
    reps = 5
    for _ in range(reps):
        b, _h = one()
    st = ek.stats()
    L.ek_set_timing(0)
    ms = st.total_kernel_ms / max(int(st.sweep_launches), 1)
    total = int(b.numpy().astype(np.uint64).sum())
    return {"workload": "C3: 2^26-sample gather(31-entry table) + scatter_add(31 u32 bins, 31 f32 bins)", "kernel_ms": ms,
            "kernel": "ek_fast_kernel<256>: per-thread private bins (integer: red.shared.add, float: LDS/FADD/STS), 9 dispatches" if int(st.fast_launches) > 0
                      else "ek_sweep_kernel<16,false,true>: shared-memory atomics for the integer bins, private float bins",
            "m_samples_per_s": n / (ms * 1e-3) / 1e6, "in_range": total,
            "roofline": {"bound": "hbm", "achieved": 4.0 * n / (ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                         "frac": 4.0 * n / (ms * 1e-3) / 1e9 / peak_gbs, "bytes_per_sample": 4.0}}


def bench_backward(ek, L, rank, world, dist, torch, local_rank, peak_gbs, width=None):
    """SURVEY 8d C4: 80 levels x 128 nodes, node width 131072, 2 in-edges per non-leaf node to random
    nodes of the previous level, materialised fp32 weights U(0.5,1.5) with 1% exact zeros, loss = hsum
    over the last level.  Algorithmic traffic: weights once + adjoints written once and read once per
    out-edge (10.0 B / edge-adjoint).  Timed: backward() only (the tape is built once)."""
    from enoki_b200 import Float32, UInt32, fmadd, select
    F32 = ek.EK_FLOAT32
    L.ek_tape_set_graph_simplification(F32, 0)      # C4 is defined on materialised weights (SURVEY 8d)
    Lv, K, w = C4["levels"], C4["per_level"], (width or C4["width"])
    rng = np.random.default_rng(1234 + rank)
    idx = UInt32.arange(w)
    ids = [[0] * K for _ in range(Lv)]
    keep = []
    n_edges = 0
    one = Float32(1.0)
    for lvl in range(Lv):
        for k in range(K):
            if lvl == 0:
                ids[lvl][k] = L.ek_tape_append_leaf(F32, w)
                continue
            node = L.ek_tape_append_node(F32, w, b"n")
            ids[lvl][k] = node
            for p in sorted(rng.choice(K, 2, replace=False)):
                seed = int(rng.integers(1, 2**31))
                h = idx * np.uint32(2654435761) + np.uint32(seed)
                h = (h ^ (h >> 15)) * np.uint32(2246822519)
                wt = fmadd(Float32((h >> 8)), Float32(1.0 / (1 << 24)), Float32(0.5))
                wt = select((h & np.uint32(127)) < UInt32(1), Float32(0.0), wt)     # ~1% exact zeros
                keep.append(wt)
                assert L.ek_tape_append_edge(F32, ids[lvl - 1][int(p)], node, wt.index) == 0
                n_edges += 1
        ek.cuda_eval()          # materialise this level's weights (keeps the trace small)
    loss = L.ek_tape_append_node(F32, 1, b"loss")
    for k in range(K):
        assert L.ek_tape_append_edge(F32, ids[Lv - 1][k], loss, one.index) == 0
    ek.cuda_sync()
    n_nodes = Lv * K

    def run(free):
        assert L.ek_tape_backward(F32, loss, int(free)) == 0, L.ek_last_error()

    run(False); run(False)
    ek.cuda_sync()
    steps = 5
    L.ek_stats_reset()
    L.ek_timer_start()
    t_host0 = time.perf_counter()
    for _ in range(steps):
        run(False)
    host_ms = (time.perf_counter() - t_host0) * 1e3 / steps     # host time to describe + enqueue one backward()
    ms = L.ek_timer_stop()
    st = ek.stats()
    if dist is not None:
        tt = torch.tensor([ms], device=f"cuda:{local_rank}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    ms_per = ms / steps
    edge_adjoints = int(st.edge_adjoints) // steps
    # kernel-only time of the adjoint launches (per-launch CUDA events; serialises host and device)
    L.ek_set_timing(1); L.ek_stats_reset()
    run(False)
    kern_ms = ek.stats().total_kernel_ms
    L.ek_set_timing(0)
    # reachable sub-graph only: the runtime counts exactly the (edge, element) pairs it processed
    bytes_alg = 10.0 * edge_adjoints
    res = {"metric": "M edge-adjoints/s (backward)", "value": world * edge_adjoints / (ms_per * 1e-3) / 1e6,
           "unit": "M edge-adjoints/s", "ms_per_backward": ms_per, "nodes": n_nodes + 1, "edges": n_edges + K,
           "edge_adjoints_per_backward": edge_adjoints, "node_width": w,
           "roofline": {"bound": "hbm", "achieved": bytes_alg / (ms_per * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                        "frac": bytes_alg / (ms_per * 1e-3) / 1e9 / peak_gbs, "bytes_per_edge_adjoint": 10.0,
                        "weights_only_frac": 4.0 * edge_adjoints / (ms_per * 1e-3) / 1e9 / peak_gbs,
                        "note": "whole backward() incl. host scheduling and 80 per-level launches"},
           "launches_per_backward": int(st.adjoint_launches) // steps, "host_enqueue_ms": host_ms, "adjoint_kernels_ms_sum": kern_ms,
           "adjoint_kernels_frac": bytes_alg / (kern_ms * 1e-3) / 1e9 / peak_gbs}
    # final pass frees the graph; leaf gradients stay readable
    run(True)
    g = L.ek_tape_gradient(F32, ids[0][0])
    if g:
        L.ek_inc_ref_ext(g)
        res["leaf0_grad_checksum"] = float(Float32.from_index(g).numpy()[:1024].astype(np.float64).sum())
    for lvl in range(Lv):
        for k in range(K):
            L.ek_tape_dec_ref_ext(F32, ids[lvl][k])
    L.ek_tape_dec_ref_ext(F32, loss)
    del keep
    return res


if __name__ == "__main__":
    main()
