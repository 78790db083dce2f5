#!/usr/bin/env python
"""bench.py — headline benchmark of the partitioned-convolution hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload metric|ir120|...]
                  [--dump-outputs DIR]

Metric: M stereo frames / s ("Msamples/sec stereo conv @ IR=10s/48kHz block=512"): two
independent mono convolutions (LL, RR — src/dsp/StereoConvolver.cpp:35-36) with their own
480 000-tap IR each, uniform partitions of 512 (P = 938).  One "step" = one pass of the hot
path (forward FFT of every block, FDL complex-MAC sweep, inverse FFT + overlap-add) over a batch
of T = 112 608 blocks (57.7 M frames = 20 min of audio) of synthetic white noise; the job is the same
at every N ("strong" scaling).

* value            device-resident throughput (input/output already in HBM), CUDA events on the
                   engine's stream, max over ranks, L2 flushed between steps.
* e2e              same metric through the host-pointer C ABI with pinned HOST buffers (H2D + D2H in
                   the timed region, wall clock around the synchronous call, max over ranks).
* roofline         dominant kernel = the FDL sweep in the form the engine chose (b200conv_last_sweep_variant):
                   - k_tc_sweep (launch groups >= 4096 blocks, P <= 961 — the metric shape): tcgen05 kind::tf32 block-Toeplitz
                     GEMMs with the 3xTF32 split; bound "tensor": EXECUTED tf32 flops / the whole sweep stage (time lines +
                     MMAs + merge) vs half the measured bf16 rate of MEASURED_PEAKS.json; the direct-form-equivalent FP32 rate
                     against the CUDA-core FMA peak is the labelled secondary `useful_fp32_equivalent`;
                   - k_cmac_batch2 (--variant 22, shorter groups, longer IRs): every H[p][k] stays in registers for 16
                     blocks, bound "fp32": FP32 TFLOP/s vs 148 SM x 128 lanes x 2 x sm_max_mhz.
                   The SURVEY 8(d) algorithmic-bytes ratio (> 1 by construction) is the labelled secondary `hbm_algorithmic`.
                   `traffic` = dram bytes of one launch from a LIVE ncu capture of this very script
                   (--probe mode, subprocess), null when ncu / the counters are not available.
* roofline_stream  the memory-bound form of the same sweep (one block per launch, 120 s IR, working set
                   beyond L2): this is the kernel whose "% of HBM peak" is a bandwidth statement.
* parity           output of this run checked against the reference CPU convolver (oracle/_ref) on windows
                   of the stream and, for N > 1, against an unsharded single-GPU engine on rank 0; the run
                   exits non-zero above 1e-5 of peak.
* ir120            config 5 (stereo, 120 s IR = 11 250 partitions), sharded by PARTITION RANGE over the
                   ranks with the fused slot exchange over NVLink (north_star's multi-GPU case), every N.
* cpu_baseline     the reference's own CPU code (oracle/_ref, unmodified sources) on this host's cores,
                   one pinned thread per core, instance memory first-touched by its own thread.

--dump-outputs DIR writes the output the last timed step returned to its caller (the device array y[c][t] of the
headline workload) as DIR/y.npy, float32, shape (channels, blocks, block): every block when the output fits in
DUMP_BYTES, else the blocks of dump_blocks() (a fixed seeded sample with the first and the last block).  Inputs and
IRs are seeded, so two builds run with the same arguments can be compared output for output.

N > 1 (torchrun, one rank per GPU):
  metric shape (10 s IR, batch >> IR): TIME-SLICE sharding — every GPU holds the whole 7.7 MB convolver and
  produces one contiguous time slice of the batch; the P blocks of history in front of a slice are uploaded and
  forward-transformed only.  No collective and no exchange on the data path; every rank moves only its own
  slice over its own PCIe link (shared, page-locked host buffers).
  120 s IR: partition-range shards + slot exchange (see `ir120`).
"""
from __future__ import annotations

import argparse
import json
import mmap
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# one hardware queue per stream: the engine's flag barriers spin on s_post while s_main keeps launching sweeps
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

TOL = 1e-5
WORKLOADS = {
    # name: (channels, ir seconds, sample rate, block)
    "metric": dict(C=2, ir_s=10, sr=48000, block=512, desc="stereo 48 kHz, 10 s IR (480000 taps), uniform block 512"),
    "ir1": dict(C=1, ir_s=1, sr=48000, block=512, desc="mono 48 kHz, 1 s IR, uniform block 512 (config 1)"),
    "ch8": dict(C=8, ir_s=10, sr=48000, block=512, desc="8-channel 48 kHz, 10 s IR per channel, block 512 (config 4)"),
    "ir120": dict(C=2, ir_s=120, sr=48000, block=512, desc="stereo 48 kHz, 120 s IR, uniform block 512 (config 5)"),
    # two-stage shapes (head block = `block`, tail block = `tail`): not bench lines of the contract, kept for tuning runs
    "cfg2": dict(C=2, ir_s=5, sr=48000, block=128, tail=8192, desc="stereo 48 kHz, 5 s IR, two-stage head 128 / tail 8192 (config 2)"),
    "cfg3": dict(C=2, ir_s=30, sr=96000, block=64, tail=8192, desc="stereo 96 kHz, 30 s IR, two-stage head 64 / tail 8192 (config 3)"),
}
# 112608 blocks (57.7 M frames = 20 min of stereo audio per step): the sweep grid (16 bin tiles x ceil(blocks/64) x
# 2 channels, 444 CTAs resident) is 126.8 / 63.4 / 31.7 / 15.9 waves for 1 / 2 / 4 / 8 time slices (a slice sweeps one
# block more than it outputs: the overlap state of its first block) — no nearly-empty last wave at any N, and the
# per-call fixed costs of a slice (history upload + transforms, pipeline fill of the PCIe path) stay small at N = 8
T_METRIC = 112608
T_IR120 = 7104
DUMP_BYTES = 32 << 20          # --dump-outputs: at most this much of the step output (the metric's is 461 MB)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured"
    return 6650.0, 1965.0, "fallback"


def measured_bf16_peaks():
    """(burst, sustained) dense bf16 TFLOP/s of MEASURED_PEAKS.json, else the B200_PROFILING.md fallback"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        if "bf16_tflops" in d:
            return float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"]))
    return 1590.0, 1590.0


def algorithmic_bytes_per_channel_block(P: int, block: int) -> int:
    K = block + 1
    return 16 * P * K + 8 * K + 16 * block


def dump_blocks(T: int, C: int, block: int) -> np.ndarray:
    """Block indices of the step output --dump-outputs writes: all T blocks when they fit in DUMP_BYTES, else a fixed
    seeded sample of that size that includes the first and the last block (sorted)."""
    S = DUMP_BYTES // (C * block * 4)
    if T <= S:
        return np.arange(T)
    mid = np.random.default_rng(T).choice(np.arange(1, T - 1), S - 2, replace=False)
    return np.sort(np.concatenate([[0, T - 1], mid]))


def slice_plan(T: int, P: int, rank: int, count: int):
    """mirror of plan_slice() in engine.cu: (a, b, lo, tail_lo) in blocks"""
    per = -(-T // count)
    a, b = min(T, rank * per), min(T, (rank + 1) * per)
    if b <= a:
        a = b = lo = max(0, T - P)
        return a, b, lo, a
    return a, b, max(0, a - P), max(b, T - P)


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, line in self.rows:
            if t0 is not None and not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed steps + 0.6 s continuation of the same step loop"}


# ---------------------------------------------------------------------------------------------
# CPU reference timing (oracle/_ref = the unmodified reference sources; falls back to the C port)
# ---------------------------------------------------------------------------------------------
def cpu_reference_run(wl, seconds_target: float, threads: int, single_thread_leg: bool = False):
    """`threads` independent C-channel instances of the reference's uniform FFTConvolver, one per host core.
    Every worker thread pins itself to its core FIRST and then creates + clears its own instances, so that the
    15 MB of spectra / delay line it streams per block live on its own NUMA node (first touch) — with the
    instances created by the main thread all of them sat on one node and 128 threads ran 1.35x one thread."""
    from oracle import oracle as orc
    kind = "reference" if orc.ref_available() else "port"
    cls = orc.RefUniform if kind == "reference" else orc.OracleUniform
    C, block = wl["C"], wl["block"]
    L = wl["ir_s"] * wl["sr"]
    irs = [orc.synth_ir(L, c) for c in range(C)]
    cpus = sorted(os.sched_getaffinity(0))
    threads = max(1, min(threads, len(cpus)))
    phase = threading.Barrier(threads + 1)
    cmd = {"nblk": 0, "xs": None, "quit": False}
    done = [0.0] * threads
    errors = []

    def worker(i):
        try:
            try:
                os.sched_setaffinity(0, {cpus[i % len(cpus)]})       # this thread only
            except OSError:
                pass
            convs = []
            for c in range(C):
                k = cls()
                k.init(block, irs[c])
                k.clear()                # zero-fills (= first-touches) the whole frequency-domain delay line
                convs.append(k)
            while True:
                phase.wait()                                          # command published
                if cmd["quit"]:
                    return
                for c in range(C):       # channels serially on one thread, as StereoConvolver::process does
                    convs[c].run(cmd["xs"][c], block)
                done[i] = time.perf_counter()
                phase.wait()                                          # results in
        except Exception as ex:          # pragma: no cover
            errors.append(ex)
            phase.abort()

    ths = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(threads)]
    for th in ths:
        th.start()

    def run_all(nblk):
        cmd["nblk"] = nblk
        cmd["xs"] = [orc.synth_input(nblk * block, c) for c in range(C)]
        phase.wait()
        t0 = time.perf_counter()
        phase.wait()
        return max(done) - t0

    try:
        run_all(16)                      # warm-up
        cal = 8
        per_block = run_all(cal) / cal   # calibrated with ALL threads running (the sweep is memory-bound)
        nblk = int(max(16, min(16384, seconds_target / max(per_block, 1e-9))))
        dt = run_all(nblk)
    finally:
        cmd["quit"] = True
        try:
            phase.wait()
        except threading.BrokenBarrierError:
            pass
    if errors:
        raise errors[0]
    single = None
    if single_thread_leg:               # "as the plugin does it": ONE thread, the C channels serially
        convs = []
        for c in range(C):
            k = cls()
            k.init(block, irs[c])
            k.clear()
            convs.append(k)
        xs1 = [orc.synth_input(64 * block, c) for c in range(C)]
        for c in range(C):
            convs[c].run(xs1[c][:8 * block], block)
        t1 = time.perf_counter()
        for c in range(C):
            convs[c].run(xs1[c], block)
        single = 64 * block / (time.perf_counter() - t1) / 1e6
    frames = nblk * block * threads
    return {
        "value": frames / dt / 1e6, "unit": "M stereo frames/s" if C == 2 else f"M {C}-channel frames/s",
        "cores": threads, "kind": kind,
        "sample": f"{threads} independent {C}-channel instances x {nblk} blocks of {block} (one pinned thread per core, "
                  f"NUMA-local first touch, ctypes with the GIL released), uniform FFTConvolver, {wl['desc']}",
        "seconds": dt, "parallel_ms_per_block": per_block * 1e3,
        "single_thread_value": single,
    }


# ---------------------------------------------------------------------------------------------
# live DRAM-traffic capture: this script re-run under ncu in --probe mode (one kernel, one launch)
# ---------------------------------------------------------------------------------------------
PROBE_VARIANT = 0      # --variant of the run, handed to the traffic probe


def ncu_traffic(which: str, kernel_regex: str, skip: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the kernel; None (+ reason) if unavailable."""
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--print-units", "base",
           "-k", f"regex:{kernel_regex}", "-s", str(skip), "-c", "1", "--csv",
           sys.executable, os.path.abspath(__file__), "--probe", which]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, B200CONV_BENCH_VARIANT=str(PROBE_VARIANT)))
    except Exception as ex:
        return None, f"ncu failed: {type(ex).__name__}"
    tot, seen = 0.0, 0
    for line in out.stdout.splitlines():
        if "dram__bytes_" in line:
            f = [x.strip('"') for x in line.split('","')]
            try:
                tot += float(f[-1].replace(",", ""))
                seen += 1
            except Exception:
                pass
    if seen < 2:
        why = "ERR_NVGPUCTRPERM" if "ERR_NVGPUCTRPERM" in out.stdout + out.stderr else "no counter rows"
        return None, f"ncu capture gave nothing ({why})"
    return int(tot), "live ncu capture of this script (--probe), dram__bytes_read.sum + dram__bytes_write.sum, one launch"


def probe_main(which: str):
    """Minimal workload for the ncu capture: the same launches as the timed loop, nothing else."""
    import torch
    from reevr_b200.convolver import Engine
    from reevr_b200.synth import synth_input, synth_ir
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    if which == "batch":
        wl = WORKLOADS["metric"]
        C, block, T = wl["C"], wl["block"], T_METRIC
        eng = Engine(C, device=0, max_batch_blocks=T + 1, cmac_variant=int(os.environ.get("B200CONV_BENCH_VARIANT", "0")))
        assert eng.init_uniform(block, [synth_ir(wl["ir_s"] * wl["sr"], c) for c in range(C)])
        n = T * block
        x = torch.from_numpy(np.stack([synth_input(n, c) for c in range(C)])).cuda()
        y = torch.empty_like(x)
        for _ in range(4):
            flush.zero_()
            eng.process_device(x.data_ptr(), n, y.data_ptr(), n, n, sync=True)
    else:
        wl = WORKLOADS["ir120"]
        C, block = wl["C"], wl["block"]
        eng = Engine(C, device=0)
        assert eng.init_uniform(block, [synth_ir(wl["ir_s"] * wl["sr"], c) for c in range(C)])
        xs = torch.from_numpy(np.stack([synth_input(block * 16, c) for c in range(C)])).cuda()
        y = torch.empty((C, block), device="cuda")
        for i in range(12):
            eng.process_device(xs[:, i * block:].data_ptr(), xs.shape[1], y.data_ptr(), block, block, sync=True)
    eng.close()
    return 0


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="metric", choices=sorted(WORKLOADS))
    ap.add_argument("--blocks", type=int, default=0, help="blocks per step (0 = auto)")
    ap.add_argument("--variant", type=int, default=0, help="CMAC kernel variant (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-stream", dest="no_stream", action="store_true", help="skip the streaming-kernel HBM roofline and real-time legs")
    ap.add_argument("--no-traffic", dest="no_traffic", action="store_true", help="skip the live ncu DRAM-traffic captures")
    ap.add_argument("--no-ir120", dest="no_ir120", action="store_true", help="skip the config-5 (120 s IR) leg")
    ap.add_argument("--no-parity", dest="no_parity", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="print a per-variant timing table to stderr")
    ap.add_argument("--mgpu", default="p2p", choices=["p2p", "nccl"], help="partition-range shards (120 s IR): exchange path")
    ap.add_argument("--metric-shards", dest="metric_shards", default="time", choices=["time", "partition"],
                    help="N > 1, metric shape: time-slice sharding (default) or partition-range shards")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="write the output of the last timed step as DIR/y.npy (float32, seeded sample of at most "
                         f"{DUMP_BYTES >> 20} MB)")
    ap.add_argument("--probe", default=None, choices=["batch", "stream"], help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200 (the reference arm sizes its work by timing, its output is not fixed)")
    if args.probe:
        return probe_main(args.probe)
    global PROBE_VARIANT
    PROBE_VARIANT = args.variant

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = dict(WORKLOADS[args.workload])
    warm = max(args.warmup, 3)

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = len(os.sched_getaffinity(0))
        # each step = one bounded sample; keep the whole run within a few minutes
        vals = []
        for i in range(warm + args.steps):
            r = cpu_reference_run(wl, seconds_target=2.0 if i < warm else 6.0, threads=threads)
            if i >= warm:
                vals.append(r)
        v = statistics.mean(x["value"] for x in vals)
        last = vals[-1]
        line = {
            "impl": "reference", "metric": "stereo partitioned-convolution throughput (IR 10 s @ 48 kHz, block 512)",
            "value": v, "unit": "M stereo frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": warm,
            "ms_per_step": 1e3 * statistics.mean(x["seconds"] for x in vals), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "engine": "reference CPU FFTConvolver (oracle/_ref)", "threads": last["cores"]},
            "cpu_baseline": {"value": v, "unit": "M stereo frames/s", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
            "e2e": {"value": v, "unit": "M stereo frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    import ctypes
    import torch
    import torch.distributed as dist
    from reevr_b200 import _lib
    from reevr_b200.convolver import Engine
    from reevr_b200.distributed import attach_p2p, attach_reduce
    from reevr_b200.synth import synth_input, synth_ir

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fall-back)")
    lib = _lib.default()
    torch.cuda.set_device(local)
    # Pinned staging buffers must live on the NUMA node the GPU hangs off, otherwise every H2D / D2H of the
    # e2e path crosses the socket interconnect: run this process on the GPU's CPU-affinity set while the
    # buffers are allocated and first touched.
    all_cpus = os.sched_getaffinity(0)
    numa_note = "not bound"
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (max(all_cpus) // 64) + 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(hnd, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1} & all_cpus
        if cpus:
            os.sched_setaffinity(0, cpus)
            numa_note = f"process bound to the GPU's {len(cpus)} local CPUs for pinned allocations"
    except Exception as ex:       # best effort
        numa_note = f"not bound ({type(ex).__name__})"
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")   # > 126 MB L2
    hbm_peak, sm_mhz, peak_kind = measured_peaks()
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    bf16_peak, bf16_sustained = measured_bf16_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- host buffers: ONE page-locked region all ranks see (memfd + cudaHostRegister) so that every GPU can
    #      read its input slice from, and write its output slice into, the caller's buffers directly
    keep_alive = []
    registered = []          # (address, mmap, fd) of the shared page-locked regions: unregistered before exit

    def host_buffers(shape, tag):
        """returns (np array, shared?) — all ranks agree on `shared`"""
        nbytes = int(np.prod(shape)) * 4
        arr, ok = None, 1
        if world > 1:
            try:
                obj = [None]
                if rank == 0:
                    fd = os.memfd_create(f"b200conv_{tag}")
                    os.ftruncate(fd, nbytes)
                    obj = [(os.getpid(), fd)]
                dist.broadcast_object_list(obj, src=0)
                if rank != 0:
                    fd = os.open(f"/proc/{obj[0][0]}/fd/{obj[0][1]}", os.O_RDWR)
                mm = mmap.mmap(fd, nbytes)
                arr = np.frombuffer(mm, dtype=np.float32).reshape(shape)
                # (no first touch here: every rank touches its OWN time slice below, while it is bound to its GPU's
                #  CPUs, so that the pages each GPU DMAs from / into live on that GPU's NUMA node)
                if os.environ.get("B200CONV_BENCH_NO_SHARED"):
                    ok = 0
                elif lib.b200conv_register_host(arr.ctypes.data, nbytes) != 0:
                    ok = 0
                else:
                    registered.append(arr.ctypes.data)
                keep_alive.append((mm, fd))
            except Exception as ex:
                print(f"[bench] rank {rank}: shared host buffer failed ({type(ex).__name__}: {ex})", file=sys.stderr)
                ok = 0
            t = torch.tensor([ok], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok = int(t.item())
        if world == 1 or not ok:
            t = torch.empty(shape, dtype=torch.float32).pin_memory()
            keep_alive.append(t)
            return t.numpy(), False
        return arr, True

    def ptrs(a):
        return (ctypes.c_void_p * a.shape[0])(*[a[c].ctypes.data for c in range(a.shape[0])])

    def time_steps(step, steps, stream, with_clocks, frames, after_timed=None):
        """`after_timed` runs right after the last timed step, before anything else touches the output"""
        for _ in range(warm):
            step()
        barrier()
        sampler = ClockSampler(local) if (with_clocks and rank == 0) else None
        if sampler:
            sampler.start()
            time.sleep(0.3)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        t_w0 = time.perf_counter()
        for i in range(steps):
            flush.zero_()                       # evict L2 between timed iterations
            barrier()
            ev[i][0].record(stream)
            step()
            ev[i][1].record(stream)
        barrier()
        t_w1 = time.perf_counter()
        if after_timed:
            after_timed()
        ms_per_step = allmax(sum(a.elapsed_time(b) for a, b in ev)) / steps
        if with_clocks:
            # K short steps give nvidia-smi (>= 20 ms per sample) almost nothing to see: EVERY rank keeps the very
            # same step loop running for another ~0.6 s (untimed; identical count on all ranks) so that the clock /
            # throttle record of rank 0 is meaningful
            n_extra = int(min(2000, max(1, 600.0 / max(ms_per_step, 0.05))))
            for _ in range(n_extra):
                step()
            barrier()
            t_w1 = time.perf_counter()
        clocks = sampler.stop(t_w0, t_w1) if sampler else None
        return ms_per_step, frames / (ms_per_step * 1e-3) / 1e6, clocks

    def sweep_roofline(eng, run_sync, C, block, Ploc, blocks_swept, stages_all, n_frames):
        """CUDA events around every FDL-sweep launch (separate pass) -> roofline object of the dominant kernel"""
        eng.set_timing(True)
        cm_ms, cm_n, fft_ms, ifft_ms = 0.0, 0, 0.0, 0.0
        reps = 3
        for _ in range(reps):
            flush.zero_()
            barrier()
            run_sync()
            tm = eng.last_timing()
            cm_ms += tm["cmac_ms"]; cm_n += tm["cmac_launches"]; fft_ms += tm["fft_ms"]; ifft_ms += tm["ifft_ms"]
        eng.set_timing(False)
        per_launch_ms = cm_ms / max(cm_n, 1)
        blocks_per_launch = blocks_swept * reps / max(cm_n, 1)
        if len(stages_all) == 1:
            alg_bytes_launch = algorithmic_bytes_per_channel_block(Ploc, block) * C * blocks_per_launch
            ffma = 4.0 * Ploc * block * C * blocks_per_launch      # 4 FP32 FMA per complex MAC, B bins per row
        else:   # multi-stage: SURVEY 8d, sum over stages of the per-sample figures, spread over the sweep launches
            per_sample = sum(algorithmic_bytes_per_channel_block(int(x["p_end"]) - int(x["p_begin"]), int(x["block"])) / int(x["block"])
                             for x in stages_all)
            alg_bytes_launch = per_sample * C * n_frames * reps / max(cm_n, 1)
            ffma = sum(4.0 * (int(x["p_end"]) - int(x["p_begin"])) for x in stages_all) * C * n_frames * reps / max(cm_n, 1)
        fp32_tflops = 2.0 * ffma / (per_launch_ms * 1e-3) / 1e12
        hbm_alg = alg_bytes_launch / (per_launch_ms * 1e-3) / 1e9
        if eng.last_sweep_variant() == 40 and len(stages_all) == 1:
            # tensor-core sweep (kernels_tc.cuh): the timed stage is k_tc_split_x + k_tc_sweep + k_tc_merge_y.  Executed
            # tensor flops = tiles x K chunks x 24 MMAs (3xTF32 x 2 time lines x 4 k-steps) x 2*128*128*8.
            q = (max(Ploc - 1, 0) + 63) // 64 * 64
            nchunk = q // 32 + 2
            ntile = -(-(-(-int(round(blocks_per_launch)) // 64)) // 128)
            mma_flop = float(C * block * ntile * nchunk * 24) * 2.0 * 128 * 128 * 8
            tf32_peak = bf16_peak / 2.0
            tflops = mma_flop / (per_launch_ms * 1e-3) / 1e12
            return {
                "kernel": "k_tc_sweep (tcgen05.mma kind::tf32, 3xTF32 block-Toeplitz FDL sweep) incl. k_tc_split_x / k_tc_merge_y",
                "bound": "tensor", "achieved": tflops, "peak": tf32_peak, "unit": "TFLOP/s", "frac": tflops / tf32_peak,
                "peak_source": f"half of MEASURED_PEAKS.json bf16_tflops ({peak_kind}): kind::tf32 issues at half the bf16 rate "
                               "(tools/tc_probe.cu: 64 cycles per 128x128x8 MMA = 4096 flop/clk/SM)",
                "frac_of_sustained_peak": tflops / (bf16_sustained / 2.0),
                "launch_ms": per_launch_ms, "blocks_per_launch": blocks_per_launch, "partitions": Ploc,
                "flop_per_launch": mma_flop, "traffic": None,
                "useful_fp32_equivalent": {"achieved": fp32_tflops, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32_tflops / fp32_peak,
                                           "note": "4 FP32 FMA per complex MAC of the direct form / the same time, against the CUDA-core "
                                                   "FMA peak the packed-FMA sweep (cmac_variant 22, frac 0.83) is bounded by"},
                "hbm_algorithmic": {"achieved": hbm_alg, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_alg / hbm_peak,
                                    "algorithmic_bytes_per_launch": alg_bytes_launch,
                                    "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                                    "note": "SURVEY 8d streaming-form bytes / launch time; > 1 because nothing is streamed per block"},
                "step_share": {"cmac_ms": cm_ms / reps, "fft_ms": fft_ms / reps, "ifft_ms": ifft_ms / reps},
            }
        return {
            "kernel": "k_cmac_batch2 (batched FDL sweep, FFMA2)", "bound": "fp32",
            "achieved": fp32_tflops, "peak": fp32_peak, "unit": "TFLOP/s", "frac": fp32_tflops / fp32_peak,
            "peak_source": f"148 SM x 128 FMA lanes/clk x 2 flop x {sm_mhz:.0f} MHz (MEASURED_PEAKS.json sm_max_mhz, {peak_kind})",
            "launch_ms": per_launch_ms, "blocks_per_launch": blocks_per_launch, "partitions": Ploc,
            "flop_per_launch": 2.0 * ffma, "traffic": None,
            "why_fp32": "every H[p][k] is kept in registers for 16 consecutive blocks, so DRAM / L2 traffic per complex MAC is "
                        ">= 16x below the streaming form; the kernel issues exactly 4 FP32 FMA (2 FFMA2) per complex MAC",
            "hbm_algorithmic": {"achieved": hbm_alg, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_alg / hbm_peak,
                                "algorithmic_bytes_per_launch": alg_bytes_launch,
                                "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                                "note": "SURVEY 8d bytes (every block streams H and the FDL once: 16*P*K + 8*K + 16*B per "
                                        "channel-block) / launch time; > 1 because the batched sweep does not stream them — "
                                        "not a bandwidth statement, see roofline_stream for the memory-bound form"},
            "step_share": {"cmac_ms": cm_ms / reps, "fft_ms": fft_ms / reps, "ifft_ms": ifft_ms / reps},
        }

    # ------------------------------------------------------------------------------------------
    def sampled_output(y_dev, C, T, block, keep=None):
        """the dump_blocks() sample of a (C, T * block) device output; blocks outside [keep) are zeroed"""
        blocks = dump_blocks(T, C, block)
        y = y_dev.view(C, T, block).index_select(1, torch.from_numpy(blocks).to(y_dev.device))
        if keep is not None:
            y[:, (blocks < keep[0]) | (blocks >= keep[1])] = 0.0
        return y

    def run_single_or_partition(wl, T, steps, with_e2e, with_clocks, with_parity, tag, want_dump=False):
        """world == 1: the unsharded engine.  world > 1: partition-range shards (+ slot exchange / NCCL reduce)."""
        from oracle import refcheck as rc
        C, block = wl["C"], wl["block"]
        L = wl["ir_s"] * wl["sr"]
        n = T * block
        # sharded: launch groups of 7104 blocks so that exchange + inverse FFT of group i overlap the sweep of group i+1
        groups = 1 if world == 1 else max(1, round(T / 7104))
        gb = (T + groups - 1) // groups
        eng = Engine(C, device=local, max_batch_blocks=gb + 1, shard_rank=rank, shard_count=world, cmac_variant=args.variant)
        irs = [synth_ir(L, c) for c in range(C)]
        t_init = time.perf_counter()
        if "tail" in wl:
            assert eng.init_twostage(block, wl["tail"], irs)
        else:
            assert eng.init_uniform(block, irs)
        t_init = time.perf_counter() - t_init
        st = eng.stages()[0]
        P = int(st["partitions"])
        Ploc = int(st["p_end"]) - int(st["p_begin"])
        stream = torch.cuda.ExternalStream(eng.stream, device=dev)
        mgpu_path = "single GPU"
        if world > 1:
            attach_reduce(eng, device=local)          # NCCL reduce hook (always installed)
            mgpu_path = "partition-range shards + NCCL reduce of partial spectra to rank 0"
            if args.mgpu == "p2p":
                ok, why = attach_p2p(eng)             # fused slot exchange over NVLink peer memory (same answer on every rank)
                if ok:
                    mgpu_path = ("partition-range shards + fused slot exchange: sweep epilogue stores partial rows into "
                                 "the owner GPU's slot over NVLink, flag barrier, per-slice inverse FFT (no NCCL on the data path)")
                else:
                    print(f"[bench] slot exchange not available ({why}); using the NCCL reduce path", file=sys.stderr)
                    mgpu_path += f" (slot exchange not available: {why})"
        tx = torch.empty((C, n), dtype=torch.float32).pin_memory()
        keep_alive.append(tx)
        x_host = tx.numpy()
        for c in range(C):
            x_host[c] = synth_input(n, c)
        ty = torch.empty((C, n), dtype=torch.float32).pin_memory()
        keep_alive.append(ty)
        y_host = ty.numpy()
        x_dev = torch.from_numpy(x_host).cuda()
        y_dev = torch.empty_like(x_dev)

        def step_device():
            eng.process_device(x_dev.data_ptr(), n, y_dev.data_ptr(), n, n, sync=False)

        dump = {}

        def keep_output():      # partition-range shards: shard 0 holds the whole output
            if want_dump:
                dump["y"] = sampled_output(y_dev, C, T, block).cpu().numpy()

        launches0 = eng.launch_count
        ms_per_step, value, clocks = time_steps(step_device, steps, stream, with_clocks, n, keep_output)
        launches = eng.launch_count - launches0
        roof = sweep_roofline(eng, lambda: eng.process_device(x_dev.data_ptr(), n, y_dev.data_ptr(), n, n, sync=True),
                              C, block, Ploc, T, eng.stages(), n)
        inp, outp = ptrs(x_host), ptrs(y_host)
        e2e = None
        if with_e2e:
            for _ in range(2):
                eng.process_into(inp, outp, n)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                eng.process_into(inp, outp, n)
            torch.cuda.synchronize()
            dt = allmax(time.perf_counter() - t0)
            e2e = {"value": n * steps / dt / 1e6, "unit": "M stereo frames/s" if C == 2 else f"M {C}-channel frames/s",
                   "h2d_bytes_per_step": C * n * 4 * world, "d2h_bytes_per_step": C * n * 4,
                   "how": "b200conv_process() on pinned host buffers, wall clock, H2D / compute / D2H pipelined on separate streams"
                          + ("; every rank uploads the whole input (it recomputes the input spectra), rank 0 downloads the audio" if world > 1 else ""),
                   "numa": numa_note}
        parity = None
        if with_parity:
            # two consecutive host-pointer calls from a cleared state (the second one has the whole IR's history
            # behind it); rank 0 compares the second call's output
            eng.clear()
            barrier()
            eng.process_into(inp, outp, n)
            eng.process_into(inp, outp, n)
            barrier()
            if rank == 0:
                t_p = time.perf_counter()
                parity = {"tolerance": TOL, "reference": rc.kind(),
                          "what": "second of two consecutive calls from a cleared state (stream = the step's input twice)"}
                xx = [np.concatenate([x_host[c], x_host[c]]) for c in range(C)]
                errs = []
                nwin = 64
                wins = [T, 2 * T - nwin] if P + 1 + nwin < 4096 else [2 * T - nwin]
                for w0 in wins:
                    for c in range(C):
                        if P + 1 + nwin < 4096:
                            ref = rc.ref_window(block, irs[c], xx[c], w0, nwin)
                        else:       # long IR: sum of 32 IR-segment reference convolvers (linearity), host threads
                            ref = rc.ref_window_segmented(block, irs[c], xx[c], w0, nwin, nseg=32, threads=min(32, len(all_cpus)))
                        got = y_host[c][(w0 - T) * block:(w0 - T + nwin) * block]
                        errs.append(rc.peak_err(got, ref))
                parity["max_err_vs_ref"] = max(errs)
                parity["ref_windows_blocks"] = [[w - T, w - T + nwin] for w in wins]
                if world > 1:
                    e1 = Engine(C, device=local, max_batch_blocks=7105)
                    assert e1.init_uniform(block, irs)
                    t1 = torch.empty((C, n), dtype=torch.float32).pin_memory()
                    y1 = t1.numpy()
                    o1 = ptrs(y1)
                    e1.process_into(inp, o1, n)
                    e1.process_into(inp, o1, n)
                    e1.close()
                    parity["max_err_vs_n1"] = max(rc.peak_err(y_host[c], y1[c]) for c in range(C))
                    del t1
                parity["ok"] = bool(max(parity["max_err_vs_ref"], parity.get("max_err_vs_n1", 0.0)) <= TOL)
                parity["seconds"] = round(time.perf_counter() - t_p, 2)
            barrier()
        res = {
            "value": value, "ms_per_step": ms_per_step, "launches": int(allsum(launches)), "clocks": clocks, "e2e": e2e,
            "parity": parity, "roofline": roof, "dump": dump,
            "config": {"workload": wl["desc"], "channels": C, "ir_taps": eng.ir_len(0), "block": block, "partitions": P,
                       "blocks_per_step": T, "frames_per_step": n, "launch_groups_per_step": groups,
                       "parallelism": mgpu_path if world == 1 else f"x{world}: {mgpu_path} ({Ploc} partitions on rank 0)",
                       "l2": "flushed between timed steps (256 MB write)", "init_s": round(t_init, 4)},
        }
        eng.close()
        del x_dev, y_dev
        torch.cuda.empty_cache()
        return res

    # ------------------------------------------------------------------------------------------
    def run_time_sliced(wl, T, steps, with_e2e, with_clocks, with_parity, tag, want_dump=False):
        """world > 1, batch >> IR: every GPU holds the whole convolver and produces one time slice of the batch."""
        from oracle import refcheck as rc
        C, block = wl["C"], wl["block"]
        L = wl["ir_s"] * wl["sr"]
        n = T * block
        per = -(-T // world)
        eng = Engine(C, device=local, max_batch_blocks=per + 1, cmac_variant=args.variant)
        irs = [synth_ir(L, c) for c in range(C)]
        t_init = time.perf_counter()
        assert eng.init_uniform(block, irs)
        t_init = time.perf_counter() - t_init
        P = int(eng.stages()[0]["partitions"])
        a, b, lo, tail_lo = slice_plan(T, P, rank, world)
        # steady batch job: only rank 0 starts its slice at the beginning of a call and needs the previous call's last P
        # blocks as history; every other rank uploads its own history with each call (b200conv.h "slice_keep_tail")
        no_tail = rank > 0 and a >= P
        if no_tail:
            eng.set_option("slice_keep_tail", 0)
            tail_lo = T
        stream = torch.cuda.ExternalStream(eng.stream, device=dev)
        x_host, shared = host_buffers((C, n), tag + "_x")
        y_host, _ = host_buffers((C, n), tag + "_y") if shared else (None, False)
        if not shared:
            t = torch.empty((C, n), dtype=torch.float32).pin_memory()
            keep_alive.append(t)
            y_host = t.numpy()
        if shared:
            for c in range(C):
                x_host[c][a * block:b * block] = synth_input(n, c)[a * block:b * block]     # NUMA-local first touch
                y_host[c][a * block:b * block] = 0.0
        else:
            for c in range(C):
                x_host[c] = synth_input(n, c)
        barrier()
        x_dev = torch.from_numpy(x_host).cuda()
        y_dev = torch.zeros_like(x_dev)

        def step_device():
            eng.process_device_sliced(x_dev.data_ptr(), n, y_dev.data_ptr(), n, n, rank, world, sync=False)

        dump = {}

        def keep_output():      # every rank holds its own slice [a, b) of the output: sum the masked samples
            if want_dump:
                y = sampled_output(y_dev, C, T, block, keep=(a, b))
                dist.all_reduce(y)
                dump["y"] = y.cpu().numpy()

        launches0 = eng.launch_count
        ms_per_step, value, clocks = time_steps(step_device, steps, stream, with_clocks, n, keep_output)
        launches = eng.launch_count - launches0
        roof = sweep_roofline(eng, lambda: eng.process_device_sliced(x_dev.data_ptr(), n, y_dev.data_ptr(), n, n, rank, world, sync=True),
                              C, block, P, b - a, eng.stages(), (b - a) * block)
        inp, outp = ptrs(x_host), ptrs(y_host)
        e2e = None
        if with_e2e:
            for _ in range(2):
                eng.process_sliced_into(inp, outp, n, rank, world)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                eng.process_sliced_into(inp, outp, n, rank, world)
            torch.cuda.synchronize()
            dt = allmax(time.perf_counter() - t0)
            h2d = allsum(((a - lo) + (b - a) + (T - tail_lo)) * block * 4 * C)
            e2e = {"value": n * steps / dt / 1e6, "unit": "M stereo frames/s" if C == 2 else f"M {C}-channel frames/s",
                   "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": C * n * 4,
                   "how": "b200conv_process_sliced() on every rank with the SAME host arrays"
                          + (" (one memfd region, page-locked in every process): each GPU uploads its slice + P blocks of history "
                             "and writes its output slice straight into the caller's buffer over its own PCIe link" if shared else
                             " (private pinned copies per rank: shared page-locked region not available here)")
                          + "; wall clock, max over ranks",
                   "shared_host_buffers": shared, "numa": numa_note}
        parity = None
        if with_parity:
            eng.clear()
            barrier()
            eng.process_sliced_into(inp, outp, n, rank, world)
            barrier()
            eng.process_sliced_into(inp, outp, n, rank, world)
            barrier()
            if shared:
                y_all = y_host
            else:       # gather the slices on rank 0 (checker only)
                parts = [None] * world
                dist.all_gather_object(parts, (a, b, [np.array(y_host[c][a * block:b * block]) for c in range(C)]))
                y_all = np.zeros((C, n), np.float32)
                for pa, pb, ys in parts:
                    for c in range(C):
                        y_all[c][pa * block:pb * block] = ys[c]
            if rank == 0:
                t_p = time.perf_counter()
                parity = {"tolerance": TOL, "reference": rc.kind(),
                          "what": "second of two consecutive sliced calls from a cleared state (stream = the step's input twice)"}
                xx = [np.concatenate([x_host[c], x_host[c]]) for c in range(C)]
                nwin = 64
                a1 = slice_plan(T, P, 1, world)[0]
                wins = [T, T + a1 - nwin // 2, 2 * T - nwin]          # start of the call, across a slice boundary, end
                errs = []
                for w0 in wins:
                    for c in range(C):
                        ref = rc.ref_window(block, irs[c], xx[c], w0, nwin)
                        errs.append(rc.peak_err(y_all[c][(w0 - T) * block:(w0 - T + nwin) * block], ref))
                parity["max_err_vs_ref"] = max(errs)
                parity["ref_windows_blocks"] = [[w - T, w - T + nwin] for w in wins]
                e1 = Engine(C, device=local, max_batch_blocks=7105)
                assert e1.init_uniform(block, irs)
                t1 = torch.empty((C, n), dtype=torch.float32).pin_memory()
                y1 = t1.numpy()
                o1 = ptrs(y1)
                e1.process_into(inp, o1, n)
                e1.process_into(inp, o1, n)
                e1.close()
                parity["max_err_vs_n1"] = max(rc.peak_err(y_all[c], y1[c]) for c in range(C))
                parity["ok"] = bool(max(parity["max_err_vs_ref"], parity["max_err_vs_n1"]) <= TOL)
                parity["seconds"] = round(time.perf_counter() - t_p, 2)
                del t1
            barrier()
        res = {
            "value": value, "ms_per_step": ms_per_step, "launches": int(allsum(launches)), "clocks": clocks, "e2e": e2e,
            "parity": parity, "roofline": roof, "dump": dump,
            "config": {"workload": wl["desc"], "channels": C, "ir_taps": eng.ir_len(0), "block": block, "partitions": P,
                       "blocks_per_step": T, "frames_per_step": n, "launch_groups_per_step": 1,
                       "parallelism": f"x{world}: time-slice sharding — every GPU holds the whole convolver ({P} partitions) and convolves "
                                      f"{per} of the {T} blocks; the {P} blocks of history in front of a slice are uploaded and "
                                      "forward-transformed only; no collective, no exchange on the data path",
                       "l2": "flushed between timed steps (256 MB write)", "init_s": round(t_init, 4)},
        }
        eng.close()
        del x_dev, y_dev
        torch.cuda.empty_cache()
        return res

    T = args.blocks or (T_METRIC if args.workload == "metric" else (7104 * 512 // wl["block"] if "tail" in wl else 7104))
    sliced = world > 1 and args.metric_shards == "time" and "tail" not in wl and args.workload != "ir120"
    runner = run_time_sliced if sliced else run_single_or_partition
    main_res = runner(wl, T, args.steps, with_e2e=not args.no_e2e, with_clocks=True, with_parity=not args.no_parity, tag="m",
                      want_dump=bool(args.dump_outputs))
    extra = None
    if not args.no_ir120 and args.workload == "metric":
        try:
            r = run_single_or_partition(dict(WORKLOADS["ir120"]), T_IR120, max(2, min(3, args.steps)), with_e2e=False,
                                        with_clocks=False, with_parity=not args.no_parity, tag="i")
            extra = {"value": r["value"], "unit": "M stereo frames/s", "ms_per_step": r["ms_per_step"], "config": r["config"],
                     "fp32_frac": r["roofline"]["frac"], "sweep_launch_ms": r["roofline"]["launch_ms"],
                     "step_share": r["roofline"]["step_share"], "parity": r["parity"]}
        except Exception as ex:       # never let the secondary leg take the headline line down
            if world > 1:
                raise
            extra = {"error": f"{type(ex).__name__}: {ex}"}

    # the memory-bound form of the sweep (real-time path, one block per launch) on a working set beyond L2:
    # this is the kernel whose "% of HBM roofline" is a bandwidth statement (DESIGN.md section 4, K2s)
    stream_roof = None
    realtime = None
    if world == 1 and not args.no_stream:
        try:    # secondary legs: never let them take the headline line down
            wl5 = WORKLOADS["ir120"]
            C5, B5 = wl5["C"], wl5["block"]
            e5 = Engine(C5, device=local)
            assert e5.init_uniform(B5, [synth_ir(wl5["ir_s"] * wl5["sr"], c) for c in range(C5)])
            P5 = int(e5.stages()[0]["partitions"])
            xs5 = torch.from_numpy(np.stack([synth_input(B5 * 72, c) for c in range(C5)])).cuda()
            y5 = torch.empty((C5, B5), device="cuda")
            for i in range(8):
                e5.process_device(xs5[:, i * B5:].data_ptr(), xs5.shape[1], y5.data_ptr(), B5, B5, sync=True)
            e5.set_timing(True)
            ts5 = []
            for i in range(8, 72):
                e5.process_device(xs5[:, i * B5:].data_ptr(), xs5.shape[1], y5.data_ptr(), B5, B5, sync=True)
                ts5.append(e5.last_timing()["cmac_ms"])
            e5.close()
            t5 = statistics.median(ts5)
            bytes5 = 16 * P5 * (B5 + 1) * C5                      # every H and FDL row read once per block step
            stream_roof = {"kernel": "streaming FDL sweep (one 512-sample block per launch)", "workload": wl5["desc"],
                           "working_set_bytes": 2 * P5 * B5 * 8 * C5, "bound": "hbm", "launch_ms": t5,
                           "achieved": bytes5 / (t5 * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                           "frac": bytes5 / (t5 * 1e-3) / 1e9 / hbm_peak, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                           "algorithmic_bytes_per_launch": bytes5, "traffic": None}
        except Exception as ex:
            stream_roof = {"error": f"{type(ex).__name__}: {ex}"}
        try:    # the real-time calls a plugin makes: host pointers, one block per call, synchronous
            def latency(call, reps=300, warm_calls=50):
                for _ in range(warm_calls):
                    call()
                lat = []
                for _ in range(reps):
                    t0 = time.perf_counter()
                    call()
                    lat.append(time.perf_counter() - t0)
                lat.sort()
                return lat[len(lat) // 2] * 1e6, lat[int(0.99 * len(lat))] * 1e6
            C0, B0 = wl["C"], wl["block"]
            e0 = Engine(C0, device=local)
            assert e0.init_uniform(B0, [synth_ir(wl["ir_s"] * wl["sr"], c) for c in range(C0)])
            blk = [synth_input(B0, c) for c in range(C0)]
            med, p99 = latency(lambda: e0.process(blk))
            e0.close()
            realtime = {"call": "b200conv_process(), host pointers, len = block = 512, uniform handle of the metric shape, synchronous",
                        "median_us": med, "p99_us": p99, "value": B0 / med, "budget_us": B0 / 48000 * 1e6,
                        "unit": "M stereo frames/s" if C0 == 2 else f"M {C0}-channel frames/s"}
            # REEV-R's own shape: StereoConvolver in quad mode (LL, RR, LR, RL), two-stage head 128 / tail 8192
            # (StereoConvolver.cpp:8-31), 10 s IRs, host block 128, true-stereo mixdown on the device
            from reevr_b200.convolver import StereoConvolver
            sc = StereoConvolver(device=local)
            sc.prepare(128)
            sc.loadImpulse(*[synth_ir(480000, c) for c in range(4)])
            sc.enable_device_mixdown(true_stereo=True)
            l_, r_ = synth_input(128, 0), synth_input(128, 1)
            med2, p992 = latency(lambda: sc.process_mixed(l_, r_), reps=600, warm_calls=200)
            realtime["reevr_quad"] = {"call": "StereoConvolver quad, two-stage 128/8192, 10 s IRs, len 128, device mixdown (one call, 2 in / 2 out)",
                                      "median_us": med2, "p99_us": p992, "budget_us": 128 / 48000 * 1e6}
            sc._e.close()
            # ... and the whole reverb section of processBlock on the device: dry block + send / reverb envelopes in,
            # filters + predelay + 4 convolvers + mixdown + width + dry/wet, final mix out (b200conv_chain_process)
            ec = Engine(4, device=local)
            assert ec.init_twostage(128, 8192, [synth_ir(480000, c) for c in range(4)])
            ec.chain_configure(srate=48000.0, lowcut_hz=120.0, lowcut_slope=1, highcut_hz=8000.0, highcut_slope=2, predelay=480,
                               width=0.8, drygain=0.7, wetgain=0.7, true_stereo=True)
            ys_, yr_ = np.full(128, 0.9, np.float32), np.full(128, 0.8, np.float32)
            med3, p993 = latency(lambda: ec.chain_process(l_, r_, ys_, yr_), reps=600, warm_calls=200)
            realtime["reevr_quad_chain"] = {"call": "b200conv_chain_process: send envelope + 12/24 dB cuts + predelay + quad two-stage 128/8192 "
                                                    "+ mixdown + reverb envelope + width + dry/wet, len 128",
                                            "median_us": med3, "p99_us": p993, "budget_us": 128 / 48000 * 1e6}
            ec.close()
        except Exception as ex:
            realtime = dict(realtime or {}, error=f"{type(ex).__name__}: {ex}")

    # Not the metric's configuration, reported for orientation only: offline rendering is free to choose its partition
    # size (the output is the same linear convolution) — the same job through a uniform handle of block 8192 (P = 59)
    offline = None
    if world == 1 and not args.no_stream and args.workload == "metric":
        try:
            C0, L0 = wl["C"], wl["ir_s"] * wl["sr"]
            n0 = T * wl["block"]
            eb = Engine(C0, device=local, max_batch_blocks=n0 // 8192 + 1)
            assert eb.init_uniform(8192, [synth_ir(L0, c) for c in range(C0)])
            xb = torch.from_numpy(np.stack([synth_input(n0, c) for c in range(C0)])).cuda()
            yb = torch.empty_like(xb)
            stb = torch.cuda.ExternalStream(eb.stream, device=dev)
            for _ in range(2):
                eb.process_device(xb.data_ptr(), n0, yb.data_ptr(), n0, n0, sync=True)
            e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            flush.zero_()
            torch.cuda.synchronize()
            e0_.record(stb)
            eb.process_device(xb.data_ptr(), n0, yb.data_ptr(), n0, n0, sync=False)
            e1_.record(stb)
            torch.cuda.synchronize()
            msb = e0_.elapsed_time(e1_)
            offline = {"what": "NOT the metric configuration: the same stream and IR through a uniform handle with 8192-sample "
                               "partitions (P = 59), which a batch caller may choose freely — identical linear convolution",
                       "value": n0 / msb / 1e3, "unit": "M stereo frames/s", "ms_per_step": msb}
            eb.close()
            del xb, yb
            torch.cuda.empty_cache()
        except Exception as ex:
            offline = {"error": f"{type(ex).__name__}: {ex}"}

    if args.sweep and rank == 0 and world == 1:
        subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sweep.py"), "--blocks", str(T)], stdout=sys.stderr)

    rc_exit = 0
    if rank == 0:
        if world == 1 and not args.no_traffic and args.workload == "metric":
            tr, how = ncu_traffic("batch", "k_tc_sweep" if main_res["roofline"].get("bound") == "tensor" else "k_cmac_batch2", 2)
            main_res["roofline"]["traffic"] = tr
            main_res["roofline"]["traffic_source"] = how
            if stream_roof and "error" not in stream_roof:
                tr, how = ncu_traffic("stream", "k_cmac_stream", 9)
                stream_roof["traffic"] = tr
                stream_roof["traffic_source"] = how
        cpu = None
        os.sched_setaffinity(0, all_cpus)          # the CPU baseline uses every host core again
        if not args.no_cpu and world == 1:
            try:
                cpu = cpu_reference_run(wl, seconds_target=12.0, threads=len(all_cpus), single_thread_leg=True)
                cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "parallel_ms_per_block", "single_thread_value")}
            except Exception as ex:       # the GPU numbers stand on their own
                cpu = {"error": f"{type(ex).__name__}: {ex}"}
        C = wl["C"]
        line = {
            "metric": "stereo partitioned-convolution throughput (IR 10 s @ 48 kHz, block 512)" if args.workload == "metric"
                      else f"partitioned-convolution throughput ({wl['desc']})",
            "value": main_res["value"], "unit": "M stereo frames/s" if C == 2 else f"M {C}-channel frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": main_res["config"], "clocks": main_res["clocks"], "e2e": main_res["e2e"],
            "gpu_launches": main_res["launches"], "roofline": main_res["roofline"], "cpu_baseline": cpu,
            "parity": main_res["parity"],
            "arithmetic": ("FP32 results from tf32 tensor-core products: 3xTF32 split (hi*hi + hi*lo + lo*hi), FP32 accumulate, "
                           "chains of 48 MMAs folded into FP32 registers; same 1e-5 parity bar (see parity)"
                           if main_res["roofline"].get("bound") == "tensor" else "FP32 FMA (packed FFMA2)"),
        }
        if extra:
            line["ir120"] = extra
        if stream_roof:
            line["roofline_stream"] = stream_roof
        if realtime:
            line["realtime_process"] = realtime
        if offline:
            line["offline_block8192"] = offline
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in main_res["dump"].items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
        for name, p in (("metric", main_res["parity"]), ("ir120", (extra or {}).get("parity"))):
            if p and not p.get("ok", True):
                print(f"[bench] PARITY FAILURE ({name}): {p}", file=sys.stderr)
                rc_exit = 3
    # orderly teardown: nothing in flight, page-locked shared regions unregistered while the context is still alive
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    for addr in registered:
        lib.b200conv_unregister_host(addr)
    del flush
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return rc_exit


if __name__ == "__main__":
    sys.exit(main())
